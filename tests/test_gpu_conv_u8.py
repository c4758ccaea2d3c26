"""vn.nn.U8Conv2d on the GPU: forward and weight / bias gradient against float64, the bitwise properties of the two frame
sources, the drop-in use in a policy, launches and synchronisation, CUDA-graph replay, and guard bytes around every
output the C ABI writes."""
import ctypes as C
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
F = torch.nn.functional

vn = importlib.import_module("a2cat-vn-pytorch_b200")

pytestmark = pytest.mark.gpu

# (cin, cout, k, stride, frame side): the reference's first layer, examples/a2c_maze.py's, depth, the reference's
# native 174 x 174 frames (rows padded to 16 bytes), a small-stride 3 x 3
GEOMS = [(3, 32, 7, 4, 84), (3, 16, 8, 4, 84), (1, 32, 7, 4, 84), (3, 32, 7, 4, 174), (3, 8, 3, 1, 84)]
GEOM_IDS = ["rgb_k7s4", "rgb_k8s4", "depth_k7s4", "native174", "rgb_k3s1"]


def _batch(n, side, c, seed):
    """uint8 [n, side, side, c] with rows padded to 16 bytes (StoreLayout.batch)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pitch = (side * side * c + 15) // 16 * 16
    raw = torch.randint(0, 256, (max(n, 1), pitch), dtype=torch.uint8, device="cuda", generator=g)
    return raw.as_strided((n, side, side, c), (pitch, side * c, c, 1))


def _layer(cin, cout, k, s, bias=True, seed=0):
    torch.manual_seed(seed)
    return vn.nn.U8Conv2d(cin, cout, k, stride=s, bias=bias).cuda()


def _rel(y, y64):
    return float((y.double() - y64).abs().max() / y64.abs().max())


def _f64_forward(x, layer):
    w = layer.weight.detach().double()
    b = None if layer.bias is None else layer.bias.detach().double()
    return F.conv2d(x.permute(0, 3, 1, 2).double() / 255, w, b, layer.stride)


def _f32_forward(x, layer):
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        return F.conv2d(x.permute(0, 3, 1, 2).float() / 255, layer.weight.detach(),
                        None if layer.bias is None else layer.bias.detach(), layer.stride)
    finally:
        torch.backends.cudnn.allow_tf32 = prev


def _check(e, e_torch):
    assert e <= 1e-5 and e <= 4 * e_torch + 1e-7, (e, e_torch)


@pytest.mark.parametrize("n", [1, 7, 4096])
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_forward_matches_float64(geom, bias, n):
    cin, cout, k, s, side = geom
    if side == 174 and n == 4096:
        n = 1024   # 1,024 native frames are 93 MB of uint8 and 0.8 GB of float64 reference
    layer = _layer(cin, cout, k, s, bias, seed=n)
    x = _batch(n, side, cin, seed=n + 1)
    with torch.no_grad():
        y = layer(x)
    torch.cuda.synchronize()
    y64 = _f64_forward(x, layer)
    assert y.shape == y64.shape and y.dtype == torch.float32
    _check(_rel(y, y64), _rel(_f32_forward(x, layer), y64))


def _thor(n_envs=64):
    scene = vn.scenes.make_thor_scene(1500, (50, 60), n_goals=4, planes=("rgb", "depth", "segmentation"))
    return vn.GraphVecEnv(vn.compile_world([scene], vn.GYM_GRAPH), n_envs, seed=3, obs_layout="aux5", host_outputs=False)


@pytest.fixture(scope="module")
def env():
    e = _thor()
    e.reset()
    yield e
    e.close()


@pytest.mark.parametrize("geom", [g for g in GEOMS if g[4] == 84], ids=[i for g, i in zip(GEOMS, GEOM_IDS) if g[4] == 84])
def test_weight_gradient_matches_float64(env, geom):
    cin, cout, k, s, _ = geom
    plane = "rgb" if cin == 3 else "depth"
    dw = env.dw
    g = torch.Generator(device="cuda").manual_seed(5)
    store_t = torch.randint(0, dw.world.n_states, (20, 410), dtype=torch.int32, device="cuda", generator=g)
    states = store_t.t()                                      # [410, 20] strided view of time-major storage: 8,200 frames
    layer = _layer(cin, cout, k, s, True, seed=1)
    y = layer.forward_states(dw, states, plane)
    go = torch.randn(y.shape, device="cuda", generator=g)
    y.backward(go)
    x = dw.plane_view(plane)[states.reshape(-1).long()]       # [N, H, W, C]
    w64 = layer.weight.detach().double().requires_grad_()
    b64 = layer.bias.detach().double().requires_grad_()
    F.conv2d(x.permute(0, 3, 1, 2).double() / 255, w64, b64, s).backward(go.double().flatten(0, 1))
    w32 = layer.weight.detach().clone().requires_grad_()
    b32 = layer.bias.detach().clone().requires_grad_()
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        F.conv2d(x.permute(0, 3, 1, 2).float() / 255, w32, b32, s).backward(go.flatten(0, 1))
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    _check(_rel(layer.weight.grad, w64.grad), _rel(w32.grad, w64.grad))
    _check(_rel(layer.bias.grad, b64.grad), _rel(b32.grad, b64.grad))


def test_batch_path_equals_store_path(env):
    layer = _layer(3, 32, 7, 4)
    gen = np.random.default_rng(0)
    for _ in range(5):
        env.step(torch.as_tensor(gen.integers(0, 4, env.num_envs), dtype=torch.int32, device="cuda"))
    with torch.no_grad():
        a = layer(env.obs_buf["rgb"])
        b = layer.forward_states(env.dw, env.obs_state)
    assert torch.equal(a, b)


def test_batch_equals_its_halves_and_runs_repeat():
    layer = _layer(3, 32, 7, 4)
    x = _batch(1000, 84, 3, seed=9)
    with torch.no_grad():
        y = layer(x)
        halves = torch.cat([layer(x[:500]), layer(x[500:])])
        again = layer(x)
    assert torch.equal(y, halves) and torch.equal(y, again)


def test_backward_repeats_bitwise(env):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 300), dtype=torch.int32, device="cuda").t()
    go = torch.randn((300, 20, 32, 20, 20), device="cuda")
    grads = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        layer.forward_states(env.dw, states).backward(go)
        grads.append((layer.weight.grad.clone(), layer.bias.grad.clone()))
    assert all(torch.equal(a, b) for a, b in zip(*grads))


class _Policy(torch.nn.Module):
    def __init__(self, c1):
        super().__init__()
        self.c1 = c1
        self.c2 = torch.nn.Conv2d(16, 32, 4, stride=2)
        self.fc = torch.nn.Linear(32 * 9 * 9, 4)

    def trunk(self, h1):
        return self.fc(F.relu(self.c2(F.relu(h1))).flatten(1))


def test_drop_in_policy_gradients(env, monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    torch.manual_seed(0)
    ref = _Policy(torch.nn.Conv2d(3, 16, 8, stride=4)).cuda().double()
    fused = _Policy(torch.nn.Conv2d(3, 16, 8, stride=4)).cuda()
    fused.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    fused.c1 = vn.nn.U8Conv2d.from_conv2d(fused.c1)
    assert isinstance(fused.c1, torch.nn.Conv2d) and set(fused.state_dict()) == set(ref.state_dict())
    states = torch.randint(0, env.dw.world.n_states, (5, 64), dtype=torch.int32, device="cuda").t()
    target = torch.randn(64 * 5, 4, device="cuda", dtype=torch.float64)
    x = vn.rollout.policy_input(env.dw, states.contiguous()).flatten(0, 1).double()
    (ref.trunk(ref.c1(x)) * target).sum().backward()
    (fused.trunk(fused.c1.forward_states(env.dw, states).flatten(0, 1)) * target.float()).sum().backward()
    for (name, p), (_, q) in zip(fused.named_parameters(), ref.named_parameters()):
        e = float((p.grad.double() - q.grad).abs().max() / q.grad.abs().max())
        assert e < 1e-4, (name, e)


def _library_kernels(events):
    return [e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA]


def test_launches_and_no_synchronisation(env):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 256), dtype=torch.int32, device="cuda").t()
    go = torch.randn((256, 20, 32, 20, 20), device="cuda")
    layer.forward_states(env.dw, states).backward(go)      # warm-up (library load, shared-memory attributes)
    layer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_sync_debug_mode("error")
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y = layer.forward_states(env.dw, states)
        fwd = _library_kernels(prof.events())
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y.backward(go)
        bwd = _library_kernels(prof.events())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(fwd) == 1 and "vn_conv_u8_fwd_kernel" in fwd[0], fwd
    assert len(bwd) == 2 and "vn_conv_u8_wgrad_kernel" in bwd[0] and "vn_conv_u8_wgrad_reduce_kernel" in bwd[1], bwd


def test_cuda_graph_replay_matches_eager(env):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 128), dtype=torch.int32, device="cuda").t()
    go = torch.randn((128, 20, 32, 20, 20), device="cuda")
    y = layer.forward_states(env.dw, states)
    y.backward(go)
    eager = (y.detach().clone(), layer.weight.grad.clone(), layer.bias.grad.clone())
    del y                         # its autograd graph holds the default stream's AccumulateGrad nodes
    layer.zero_grad(set_to_none=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            layer.zero_grad(set_to_none=True)
            layer.forward_states(env.dw, states).backward(go)
        layer.zero_grad(set_to_none=True)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gy = layer.forward_states(env.dw, states)
        gy.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gy, eager[0]) and torch.equal(layer.weight.grad, eager[1]) and torch.equal(layer.bias.grad, eager[2])


def _frames_struct(x):
    n, h, w, c = x.shape
    return vn.lib.U8Frames(x.data_ptr(), x.stride(0), None, 0, 0, n, 1, h, w, c, 0)


@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_outputs_stay_inside_their_buffers(geom):
    cin, cout, k, s, side = geom
    lib = vn.lib.load()
    n = 37
    x = _batch(n, side, cin, seed=2)
    oh = (side - k) // s + 1
    guard = 4096
    canary = -12345.0

    def guarded(count):
        buf = torch.full((guard + count + guard,), canary, dtype=torch.float32, device="cuda")
        return buf, buf[guard:guard + count]

    w = torch.randn(cout * cin * k * k, device="cuda") * 0.05
    b = torch.randn(cout, device="cuda")
    outb, out = guarded(n * cout * oh * oh)
    src = _frames_struct(x)
    stream = torch.cuda.current_stream().cuda_stream
    vn.lib.check(lib.vn_conv_u8_forward(C.byref(src), w.data_ptr(), b.data_ptr(), cout, k, s, out.data_ptr(), stream))
    go = torch.randn(n * cout * oh * oh, device="cuda")
    gwb, gw = guarded(w.numel())
    gbb, gb = guarded(cout)
    nbytes = lib.vn_conv_u8_wgrad_scratch_bytes(n, cin, cout, k)
    scr = torch.full((guard * 4 + nbytes + guard * 4,), 0x5A, dtype=torch.uint8, device="cuda")
    vn.lib.check(lib.vn_conv_u8_backward(C.byref(src), go.data_ptr(), cout, k, s, gw.data_ptr(), gb.data_ptr(),
                                         scr[guard * 4:].data_ptr(), nbytes, stream))
    torch.cuda.synchronize()
    for buf, count in ((outb, out.numel()), (gwb, gw.numel()), (gbb, gb.numel())):
        assert bool((buf[:guard] == canary).all()) and bool((buf[guard + count:] == canary).all())
        assert not bool((buf[guard:guard + count] == canary).any())
    assert bool((scr[:guard * 4] == 0x5A).all()) and bool((scr[guard * 4 + nbytes:] == 0x5A).all())


def test_rejects_float_input_and_unsupported_layers():
    layer = _layer(3, 32, 7, 4)
    with pytest.raises(TypeError):
        layer(torch.zeros((2, 84, 84, 3), device="cuda"))
    for kw in (dict(padding=1), dict(dilation=2), dict(groups=1, out_channels=12), dict(kernel_size=9),
               dict(in_channels=2)):
        args = dict(in_channels=3, out_channels=32, kernel_size=7, stride=4)
        args.update(kw)
        with pytest.raises(ValueError):
            vn.nn.U8Conv2d(**args)
