"""The policy's first convolution read straight from uint8 frames (``vn.nn``).

``U8Conv2d`` replaces TransposeImage + ScaledFloatFrame (deep_rl.common.env, thor_cached_auxiliary.py:61-62) + the
model's first ``Conv2d`` (models/goal.py:36-41): ``layer(frames) == F.conv2d(frames.permute(0, 3, 1, 2).float() / 255,
weight, bias, stride)`` to fp32 accuracy, with the frames taken as uint8 ``[N, H, W, C]`` - the observation leaves of
``GraphVecEnv(scaled_float=False)`` - or as state indices read from the HBM store (``forward_states``).  No float copy of
a frame is ever written: the forward is one library kernel, the weight / bias gradient two, and what autograd keeps for
the backward is the uint8 batch or the int32 index tensor.

Mixed precision: inside ``torch.autocast("cuda", dtype=torch.float16)`` or ``bfloat16`` the layer returns that dtype and
runs one-term 16-bit tensor-core kernels, as ``nn.Conv2d`` does there: ``round_to_dtype(fp32(conv2d(x / 255,
weight.to(dtype), bias.to(dtype), stride)))``.  Pixels are exact, the weight and bias are rounded like autocast's cast, the
products are exact and accumulate in fp32, and the result is rounded once.  torch's own autocast conv also rounds
``x / 255`` to ``dtype``; this layer does not, so its results are more accurate than that and not bit-equal to it.  The
backward takes ``grad_out`` in ``dtype`` and returns fp32 gradients for the fp32 parameters; a non-finite ``grad_out``
element makes its output channel's gradients non-finite, which is what ``GradScaler`` looks for.  Outside autocast, with
any other autocast dtype, or under a nested ``autocast(enabled=False)``, the fp32 kernels run.

Aliasing rule: the frames must not change between the forward and the backward.  The library rewrites an env's
observation batch on the next ``step`` without bumping torch's version counter, so autograd cannot notice.  An update
pass therefore runs ``forward_states`` over the rollout's state indices (``buf.states[:-1].t()``), which is also the
path that keeps nothing but those indices alive until the backward.

``U8PlanesConv2d`` is the same layer over several frame planes stacked along channels: ``layer(rgb, depth) ==
F.conv2d(torch.cat([rgb, depth], 3).permute(0, 3, 1, 2).float() / 255, weight, bias, stride)`` for an RGB-D encoder, or
``layer.forward_states(dw, (states, "rgb"), (goals, "rgb"))`` for an early-fusion goal encoder, with the numerics, the
autocast behaviour and the aliasing rule above.  No float frame and no concatenated frame is written.
"""
import ctypes as C

import torch

from . import lib as L
from .rollout import _call

_LP_DTYPES = {torch.float16: L.DTYPE_F16, torch.bfloat16: L.DTYPE_BF16}


def _autocast_dtype():
    """The 16-bit dtype of an enabled CUDA autocast region, or None (fp32 kernels)."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        if dt in _LP_DTYPES:
            return dt
    return None


def _frames_of_batch(x):
    """vn_u8_frames_t of a uint8 [N, H, W, C] batch whose rows are a multiple of 16 bytes apart (StoreLayout.batch)."""
    n, h, w, c = x.shape
    if x.stride()[1:] != (w * c, c, 1):
        raise ValueError("U8Conv2d: each frame must be HWC-contiguous, got strides %s" % (x.stride(),))
    pitch = x.stride(0) if n > 1 else (h * w * c + 15) // 16 * 16
    if pitch % 16 or x.data_ptr() % 16:
        raise ValueError("U8Conv2d: frames must start on 16-byte boundaries, rows a multiple of 16 bytes apart (got a "
                         "pitch of %d bytes); StoreLayout.batch / GraphVecEnv observation leaves are" % pitch)
    return L.U8Frames(x.data_ptr(), pitch, None, 0, 0, n, 1, h, w, c, 0)


def _frame_set(frames):
    """The vn_u8_frames_t array of a plane set."""
    return (L.U8Frames * len(frames))(*frames)


def _frames_of_states(dw, states, plane):
    """vn_u8_frames_t of store plane `plane` at the records named by int32 `states` ([N] or [B, T], any strides)."""
    lay = dw.world.layout
    pi = dw.plane_index(plane)
    h, w = lay.frame_hw
    if states.dim() == 1:
        idx_t, sn, st = 1, states.stride(0), 0
    elif states.dim() == 2:
        idx_t, sn, st = states.shape[1], states.stride(0), states.stride(1)
    else:
        raise ValueError("U8Conv2d.forward_states: states must be [N] or [B, T], got %s" % (tuple(states.shape),))
    n = states.numel()
    return L.U8Frames(dw.frames.data_ptr() + lay.plane_off[pi], lay.state_pitch, states.data_ptr(), sn, st, n,
                      max(idx_t, 1), h, w, lay.channels[pi], 0)


def _entry(src, name):
    """(entry point, leading arguments, n) of ``src``: one vn_u8_frames_t (vn_conv_u8_*) or a plane set
    (vn_conv_u8_planes_*)."""
    if isinstance(src, L.U8Frames):
        return "vn_conv_u8_" + name, (C.byref(src),), src.n
    return "vn_conv_u8_planes_" + name, (src, len(src)), src[0].n


class _U8Conv(torch.autograd.Function):
    """y = conv2d(x / 255, weight, bias, stride) for uint8 frames described by ``frames_of(*sources)`` (one
    vn_u8_frames_t, or a plane set from ``_frame_set``), in float32 or in the autocast dtype the forward ran under
    (recorded for the backward).  Saves only ``sources`` (uint8 batches or index tensors) for the backward."""

    @staticmethod
    def forward(ctx, weight, bias, frames_of, stride, out_shape, *sources):
        cout, _, k, _ = weight.shape
        if not weight.is_contiguous() or (bias is not None and not bias.is_contiguous()):
            raise ValueError("U8Conv2d: weight and bias must be contiguous")
        src = frames_of(*sources)
        dtype = _autocast_dtype()
        out = torch.empty(out_shape, dtype=dtype or torch.float32, device=weight.device)
        fn, head, n = _entry(src, "forward" if dtype is None else "forward_lp")
        if n:   # an empty batch launches nothing: a freshly allocated one has a null data pointer
            dt = () if dtype is None else (_LP_DTYPES[dtype],)
            _call(weight.device, fn, *head, weight.data_ptr(), L.ptr(bias), cout, k, stride, *dt, out.data_ptr(),
                  stream_of=weight)
        ctx.save_for_backward(*sources)
        ctx.frames_of, ctx.stride, ctx.has_bias, ctx.dtype = frames_of, stride, bias is not None, dtype
        ctx.wshape = tuple(weight.shape)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        need_w, need_b = ctx.needs_input_grad[0], ctx.has_bias and ctx.needs_input_grad[1]
        rest = (None,) * (3 + len(ctx.saved_tensors))
        if not (need_w or need_b):
            return (None, None) + rest
        src = ctx.frames_of(*ctx.saved_tensors)
        cout, c, k, _ = ctx.wshape
        dev = grad_out.device
        if ctx.dtype is not None:
            grad_out = grad_out.to(ctx.dtype)  # a copy kernel only when the gradient arrives in another dtype
        grad_out = grad_out.contiguous()      # a copy kernel only when autograd hands over a non-contiguous gradient
        gw = torch.empty(ctx.wshape, dtype=torch.float32, device=dev)
        gb = torch.empty(cout, dtype=torch.float32, device=dev) if ctx.has_bias else None
        fn, head, n = _entry(src, "backward" if ctx.dtype is None else "backward_lp")
        if n == 0:
            gw.zero_()
            if gb is not None:
                gb.zero_()
        else:
            nbytes = L.load().vn_conv_u8_wgrad_scratch_bytes(n, c, cout, k)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            dt = () if ctx.dtype is None else (_LP_DTYPES[ctx.dtype],)
            _call(dev, fn, *head, grad_out.data_ptr(), *dt, cout, k, ctx.stride, gw.data_ptr(), L.ptr(gb),
                  scratch.data_ptr(), nbytes, stream_of=grad_out)
        return (gw if need_w else None), (gb if need_b else None), *rest


class _U8ConvBase(torch.nn.Conv2d):
    """The nn.Conv2d geometry both layers support; ``channels_error`` is the subclass's rule for ``in_channels``."""

    def _check_geometry(self, channels_error):
        k, s = self.kernel_size, self.stride
        why = None
        if self.padding not in ((0, 0), "valid") or self.dilation != (1, 1) or self.groups != 1:
            why = "padding, dilation and groups are not supported"
        elif k[0] != k[1] or s[0] != s[1]:
            why = "kernel and stride must be square"
        elif channels_error:
            why = channels_error
        elif not 1 <= k[0] <= 8 or not 1 <= s[0] <= k[0]:
            why = "1 <= stride <= kernel_size <= 8"
        elif self.out_channels % 8 or not 8 <= self.out_channels <= 64:
            why = "out_channels must be a multiple of 8 up to 64"
        elif self.weight.dtype != torch.float32:
            why = "the parameters must be float32"
        if why:
            raise ValueError("%s: %s" % (type(self).__name__, why))

    def _out_hw(self, h, w):
        k, s = self.kernel_size[0], self.stride[0]
        return (h - k) // s + 1, (w - k) // s + 1

    def _check_device(self, t):
        if not self.weight.is_cuda or t.device != self.weight.device:
            raise ValueError("%s: the layer and its input must be on the same CUDA device" % type(self).__name__)


class U8Conv2d(_U8ConvBase):
    """Drop-in for the model's first ``nn.Conv2d`` whose input is uint8 HWC frames (see the module docstring).

    Same constructor, parameter initialisation and ``state_dict`` keys as ``nn.Conv2d``.  Supported: 1 or 3 input
    channels, a square kernel of 1..8, stride 1..kernel (square), 8..64 output channels in steps of 8, no padding,
    dilation or groups, frames of kernel..174 pixels a side; anything else raises ``ValueError`` here.  Under
    ``torch.autocast`` with fp16 or bf16 the output has that dtype (see the module docstring for the numerics); the
    autocast state is the only switch, as for ``nn.Conv2d``."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 padding_mode="zeros", device=None, dtype=None):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, padding_mode,
                         device, dtype)
        self._check_geometry(None if in_channels in (1, 3) else "in_channels must be 1 or 3")

    @classmethod
    def from_conv2d(cls, conv):
        """A U8Conv2d with the parameters of a trained ``nn.Conv2d`` (copied, on the same device)."""
        layer = cls(conv.in_channels, conv.out_channels, conv.kernel_size, conv.stride, conv.padding, conv.dilation,
                    conv.groups, conv.bias is not None, conv.padding_mode, device=conv.weight.device,
                    dtype=conv.weight.dtype)
        layer.load_state_dict(conv.state_dict())
        return layer

    def forward(self, frames):
        """frames: uint8 CUDA ``[N, H, W, C]`` (rows a multiple of 16 bytes apart, e.g. a GraphVecEnv observation leaf)
        -> float32 ``[N, out_channels, oh, ow]`` (fp16 / bf16 under autocast with that dtype)."""
        if not torch.is_tensor(frames) or frames.dtype != torch.uint8:
            raise TypeError("U8Conv2d takes uint8 [N, H, W, C] frames, got %s" %
                            (frames.dtype if torch.is_tensor(frames) else type(frames).__name__))
        if frames.dim() != 4 or frames.shape[3] != self.in_channels:
            raise ValueError("U8Conv2d: expected [N, H, W, %d] frames, got %s" % (self.in_channels, tuple(frames.shape)))
        self._check_device(frames)
        n, h, w, _ = frames.shape
        return _U8Conv.apply(self.weight, self.bias, _frames_of_batch, self.stride[0],
                             (n, self.out_channels) + self._out_hw(h, w), frames)

    def forward_states(self, dw, states, plane="rgb"):
        """The frames of store plane `plane` at the records ``states`` (int32 ``[N]`` or ``[B, T]`` with any strides,
        e.g. ``env.obs_state`` or ``buf.states[:-1].t()``, read in place) -> float32 ``[*states.shape, out_channels,
        oh, ow]`` (fp16 / bf16 under autocast with that dtype).  As with ``vn_gather_plane``, ``states`` must hold valid record indices."""
        lay = dw.world.layout
        if lay.channels[dw.plane_index(plane)] != self.in_channels:
            raise ValueError("U8Conv2d: plane %r has %d channels, the layer takes %d"
                             % (plane, lay.channels[dw.plane_index(plane)], self.in_channels))
        if states.dtype != torch.int32 or states.device != dw.device:
            states = states.to(device=dw.device, dtype=torch.int32)
        self._check_device(states)
        shape = tuple(states.shape)
        out = _U8Conv.apply(self.weight, self.bias, lambda s: _frames_of_states(dw, s, plane), self.stride[0],
                            (states.numel(), self.out_channels) + self._out_hw(*lay.frame_hw), states)
        return out.view(shape + tuple(out.shape[1:]))


class U8PlanesConv2d(_U8ConvBase):
    """Drop-in for a first ``nn.Conv2d`` whose input is several uint8 HWC frame planes concatenated along channels in
    order, e.g. ``plane_channels=(3, 1)`` for RGB-D or ``(3, 3)`` for observation + goal (see the module docstring).

    ``in_channels = sum(plane_channels)``; parameter initialisation and ``state_dict`` keys are those of
    ``nn.Conv2d(in_channels, ...)``.  Supported: 1 to 4 planes of 1 or 3 channels, 8 channels in all, and the kernel,
    stride and output channels of ``U8Conv2d``; anything else raises ``ValueError`` here.  Frames up to 84 x 84 take
    every such set, the reference's 174 x 174 frames up to 5 channels (RGB-D); a larger frame set is rejected by the
    library.  Autocast and the aliasing rule are those of ``U8Conv2d``."""

    def __init__(self, plane_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 padding_mode="zeros", device=None, dtype=None):
        planes = tuple(int(c) for c in plane_channels)
        if not planes:
            raise ValueError("U8PlanesConv2d: 1 to 4 planes are supported, got 0")
        super().__init__(sum(planes), out_channels, kernel_size, stride, padding, dilation, groups, bias,
                         padding_mode, device, dtype)
        self.plane_channels = planes
        why = None
        if not 1 <= len(planes) <= 4:
            why = "1 to 4 planes are supported, got %d" % len(planes)
        elif any(c not in (1, 3) for c in planes):
            why = "each plane must have 1 or 3 channels, got %s" % (planes,)
        elif sum(planes) > 8:
            why = "at most 8 channels in all, got %d" % sum(planes)
        self._check_geometry(why)

    @classmethod
    def from_conv2d(cls, conv, plane_channels):
        """A U8PlanesConv2d with the parameters of a trained ``nn.Conv2d(sum(plane_channels), ...)`` (copied, on the
        same device)."""
        if sum(plane_channels) != conv.in_channels:
            raise ValueError("U8PlanesConv2d: plane_channels %s do not add up to the conv's %d input channels"
                             % (tuple(plane_channels), conv.in_channels))
        layer = cls(plane_channels, conv.out_channels, conv.kernel_size, conv.stride, conv.padding, conv.dilation,
                    conv.groups, conv.bias is not None, conv.padding_mode, device=conv.weight.device,
                    dtype=conv.weight.dtype)
        layer.load_state_dict(conv.state_dict())
        return layer

    def extra_repr(self):
        return "plane_channels=%s, %s" % (self.plane_channels, super().extra_repr())

    def forward(self, *frames):
        """One uint8 CUDA ``[N, H, W, c_i]`` batch per plane (rows a multiple of 16 bytes apart, e.g.
        ``env.obs_buf["rgb"], env.obs_buf["depth"]``) -> float32 ``[N, out_channels, oh, ow]`` (fp16 / bf16 under
        autocast with that dtype)."""
        if len(frames) != len(self.plane_channels):
            raise TypeError("U8PlanesConv2d takes %d frame batches, got %d" % (len(self.plane_channels), len(frames)))
        for x, c in zip(frames, self.plane_channels):
            if not torch.is_tensor(x) or x.dtype != torch.uint8:
                raise TypeError("U8PlanesConv2d takes uint8 [N, H, W, C] frames, got %s" %
                                (x.dtype if torch.is_tensor(x) else type(x).__name__))
            if x.dim() != 4 or x.shape[3] != c or x.shape[:3] != frames[0].shape[:3]:
                raise ValueError("U8PlanesConv2d: expected [N, H, W, c] frames with c = %s and one N, H, W, got %s"
                                 % (self.plane_channels, [tuple(f.shape) for f in frames]))
            self._check_device(x)
        n, h, w, _ = frames[0].shape
        return _U8Conv.apply(self.weight, self.bias, lambda *xs: _frame_set([_frames_of_batch(x) for x in xs]),
                             self.stride[0], (n, self.out_channels) + self._out_hw(h, w), *frames)

    def forward_states(self, dw, *sources):
        """One ``(states, plane)`` pair per plane: the frames of store plane ``plane`` at the records ``states`` (int32
        ``[N]`` or ``[B, T]`` with any strides, all of one shape, read in place; e.g. ``(buf.states[:-1].t(), "rgb"),
        (buf.goals[:-1].t(), "rgb")``) -> float32 ``[*states.shape, out_channels, oh, ow]`` (fp16 / bf16 under autocast
        with that dtype).  ``states`` must hold valid record indices."""
        if len(sources) != len(self.plane_channels):
            raise TypeError("U8PlanesConv2d.forward_states takes %d (states, plane) pairs, got %d"
                            % (len(self.plane_channels), len(sources)))
        lay = dw.world.layout
        states, planes = [], []
        for (s, plane), c in zip(sources, self.plane_channels):
            if lay.channels[dw.plane_index(plane)] != c:
                raise ValueError("U8PlanesConv2d: plane %r has %d channels, the layer takes %d there"
                                 % (plane, lay.channels[dw.plane_index(plane)], c))
            if s.dtype != torch.int32 or s.device != dw.device:
                s = s.to(device=dw.device, dtype=torch.int32)
            if s.shape != sources[0][0].shape or s.dim() not in (1, 2):
                raise ValueError("U8PlanesConv2d.forward_states: states must be [N] or [B, T] of one shape, got %s"
                                 % ([tuple(x.shape) for x, _ in sources],))
            self._check_device(s)
            states.append(s)
            planes.append(plane)
        shape = tuple(states[0].shape)
        out = _U8Conv.apply(self.weight, self.bias,
                            lambda *ss: _frame_set([_frames_of_states(dw, s, p) for s, p in zip(ss, planes)]),
                            self.stride[0], (states[0].numel(), self.out_channels) + self._out_hw(*lay.frame_hw),
                            *states)
        return out.view(shape + tuple(out.shape[1:]))
