"""Which arguments the plane-set entry points of the uint8-frame convolution (vn_conv_u8_planes_*) accept and which they
reject, with the return code and the message of each rejection.  As in test_conv_u8_arg_checks.py, a process that sees
no CUDA device runs every call: the descriptors carry aligned addresses that are never dereferenced, and a call that
passes validation fails at its first CUDA runtime call with VN_ECUDA.  Every case differs from the accepted call of its
entry point (an RGB-D set: a 3-channel and a 1-channel source, 84 x 84, (k 7, stride 4, cout 32)) in one argument."""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, -1, -2, -3
F16, BF16 = 1, 2
RGB, DEPTH = 84 * 84 * 3, 84 * 84   # frame bytes; both multiples of 16

# case -> (return code, a piece of the message it must leave); shared by every entry point
_SHARED = {
    "srcs_null": (EINVAL, "srcs is null"),
    "no_sources": (EINVAL, "0 sources"),
    "five_sources": (EUNSUPPORTED, "5 sources (1 to 4 are supported)"),
    "channels_two": (EUNSUPPORTED, "source 1: 2 channels (1 or 3 are supported)"),
    "channels_nine": (EUNSUPPORTED, "9 channels in all (at most 8 are supported)"),
    "n_mismatch": (EINVAL, "source 1: n, idx_t, h, w (8, 1, 84, 84) differ from source 0's (16, 1, 84, 84)"),
    "h_mismatch": (EINVAL, "source 1: n, idx_t, h, w (16, 1, 80, 84) differ"),
    "w_mismatch": (EINVAL, "source 1: n, idx_t, h, w (16, 1, 84, 80) differ"),
    "idx_t_mismatch": (EINVAL, "source 1: n, idx_t, h, w (16, 4, 84, 84) differ from source 0's (16, 2, 84, 84)"),
    "source1_base_null": (EINVAL, "source 1: frame base is null"),
    "source1_base_off8": (EINVAL, "source 1: frame base and pitch"),
    "source1_pitch_off8": (EINVAL, "source 1: frame base and pitch (7064) must be 16-byte aligned"),
    "source1_pitch_below_frame": (EINVAL, "source 1: pitch 7040 is less than a 84 x 84 x 1 frame"),
    "source1_n_negative": (EINVAL, "source 1: n=-1"),
    "source1_idx_t_zero": (EINVAL, "source 1: idx_t=0 does not divide n=16"),
    "kernel_9": (EUNSUPPORTED, "kernel 9, stride 4"),
    "kernel_zero": (EUNSUPPORTED, "kernel 0, stride 0"),
    "stride_above_kernel": (EUNSUPPORTED, "kernel 3, stride 4"),
    "cout_12": (EUNSUPPORTED, "12 output channels"),
    "cout_72": (EUNSUPPORTED, "72 output channels"),
    "frame_175": (EUNSUPPORTED, "175 x 175 frame with kernel 7"),
    "frame_below_kernel": (EUNSUPPORTED, "6 x 6 frame with kernel 7"),
    "native_174_six_channels": (EUNSUPPORTED, "a 174 x 174 frame set of 6 channels (181664 bytes) does not fit"),
}
# accepted everywhere (VN_ECUDA: validation passed) or launching nothing (VN_OK)
_ACCEPTED = {
    "accepted": ECUDA, "one_source": ECUDA, "four_sources_8ch": ECUDA, "obs_goal_indices": ECUDA,
    "native_174_rgbd": ECUDA, "native_174_five_channels": ECUDA, "cout_64_k8_8ch": ECUDA, "k1_s1_1ch": ECUDA,
    "n0": OK, "n0_store": OK,
}
_FWD = {"null_weight": (EINVAL, "weight and out must not be null"), "null_out": (EINVAL, "weight and out must not be null")}
_BWD = {
    "null_grad_out": (EINVAL, "grad_out and grad_weight must not be null"),
    "null_grad_weight": (EINVAL, "grad_out and grad_weight must not be null"),
    "null_scratch": (EINVAL, "scratch must be a 16-byte aligned device buffer"),
    "scratch_off8": (EINVAL, "scratch must be a 16-byte aligned device buffer"),
    "scratch_short": (EINVAL, "scratch bytes"),
}
_DTYPE = {"dtype_zero": (EUNSUPPORTED, "dtype 0 (VN_DTYPE_F16 or VN_DTYPE_BF16 are supported)"),
          "dtype_three": (EUNSUPPORTED, "dtype 3"), "dtype_minus_one": (EUNSUPPORTED, "dtype -1")}
EXPECTED = {
    "vn_conv_u8_planes_forward": dict(
        _SHARED, **_FWD, off2_weight=(EINVAL, "weight, bias and out must be 4-byte aligned"),
        off2_bias=(EINVAL, "weight, bias and out must be 4-byte aligned"),
        off2_out=(EINVAL, "weight, bias and out must be 4-byte aligned")),
    "vn_conv_u8_planes_forward_lp": dict(
        _SHARED, **_FWD, **_DTYPE, off2_weight=(EINVAL, "weight and bias must be 4-byte aligned"),
        off2_bias=(EINVAL, "weight and bias must be 4-byte aligned"), off1_out=(EINVAL, "out must be 2-byte aligned")),
    "vn_conv_u8_planes_backward": dict(
        _SHARED, **_BWD, off2_grad_out=(EINVAL, "grad_out, grad_weight and grad_bias must be 4-byte aligned"),
        off2_grad_weight=(EINVAL, "grad_out, grad_weight and grad_bias must be 4-byte aligned"),
        off2_grad_bias=(EINVAL, "grad_out, grad_weight and grad_bias must be 4-byte aligned")),
    "vn_conv_u8_planes_backward_lp": dict(
        _SHARED, **_BWD, **_DTYPE, off1_grad_out=(EINVAL, "grad_out must be 2-byte aligned"),
        off2_grad_weight=(EINVAL, "grad_weight and grad_bias must be 4-byte aligned"),
        off2_grad_bias=(EINVAL, "grad_weight and grad_bias must be 4-byte aligned")),
}
# accepted only by some entry points
_EXTRA_OK = {"vn_conv_u8_planes_forward": "no_bias", "vn_conv_u8_planes_forward_lp": "no_bias f16 off2_out odd_pixels",
             "vn_conv_u8_planes_backward": "no_grad_bias n0_no_scratch",
             "vn_conv_u8_planes_backward_lp": "no_grad_bias n0_no_scratch f16 off2_grad_out odd_pixels"}


def _entry_points(vn):
    L = vn.lib
    lib = L.load()
    addr = iter(range(2 << 32, 3 << 32, 1 << 24))

    def p():
        return next(addr)

    keep = []

    def frames(a):
        """The call's vn_u8_frames_t array: a["srcs"] is a list of per-source dicts."""
        fs = [L.U8Frames(s["base"], s["pitch"], s["idx"], s["sn"], s["st"], s["n"], s["idx_t"], s["h"], s["w"], s["c"],
                         0) for s in a["srcs"]]
        arr = (L.U8Frames * max(len(fs), 1))(*fs)
        keep.append(arr)
        return None if a["srcs_null"] else arr

    def src(base, c, **kw):
        return dict(dict(base=base, pitch=84 * 84 * c, idx=None, sn=0, st=0, n=16, idx_t=1, h=84, w=84, c=c), **kw)

    rgb, depth, goal, idx, idx2 = p(), p(), p(), p(), p()
    rgbd = [src(rgb, 3), src(depth, 1)]

    def with1(**kw):
        return dict(srcs=[rgbd[0], dict(rgbd[1], **kw)])

    def store(base, c, index, side=84):
        pitch = (side * side * 8 + 15) // 16 * 16 * 2
        return src(base, c, idx=index, pitch=pitch, sn=1, st=8, idx_t=2, h=side, w=side)

    def native(*cs):
        bases = [rgb, depth, goal, p()]
        return dict(srcs=[src(bases[i], c, h=174, w=174, pitch=(174 * 174 * c + 15) // 16 * 16)
                          for i, c in enumerate(cs)])

    accepted = dict(srcs_null=False, srcs=rgbd, cout=32, k=7, stride=4, dtype=BF16)
    cases = dict(
        srcs_null=dict(srcs_null=True), no_sources=dict(srcs=[]),
        five_sources=dict(srcs=[src(rgb, 1), src(depth, 1), src(goal, 1), src(p(), 1), src(p(), 1)]),
        channels_two=with1(c=2, pitch=RGB), channels_nine=dict(srcs=[src(rgb, 3), src(depth, 3), src(goal, 3)]),
        n_mismatch=with1(n=8), h_mismatch=with1(h=80), w_mismatch=with1(w=80),
        idx_t_mismatch=dict(srcs=[store(rgb, 3, idx), dict(store(depth, 1, idx2), idx_t=4)]),
        source1_base_null=with1(base=None), source1_base_off8=with1(base=depth + 8),
        source1_pitch_off8=with1(pitch=DEPTH + 8), source1_pitch_below_frame=with1(pitch=DEPTH - 16),
        source1_n_negative=with1(n=-1), source1_idx_t_zero=with1(idx=idx, idx_t=0),
        kernel_9=dict(k=9), kernel_zero=dict(k=0, stride=0), stride_above_kernel=dict(k=3, stride=4),
        cout_12=dict(cout=12), cout_72=dict(cout=72),
        frame_175=dict(srcs=[src(rgb, 3, h=175, w=175, pitch=175 * 175 * 3 + 13),
                             src(depth, 1, h=175, w=175, pitch=175 * 175 + 15)]),
        frame_below_kernel=dict(srcs=[src(rgb, 3, h=6, w=6, pitch=112), src(depth, 1, h=6, w=6, pitch=48)]),
        native_174_six_channels=native(3, 3),
        one_source=dict(srcs=[src(rgb, 3)]),
        four_sources_8ch=dict(srcs=[src(rgb, 3), src(depth, 3), src(goal, 1), src(p(), 1)], cout=64, k=8),
        obs_goal_indices=dict(srcs=[store(rgb, 3, idx), store(rgb, 3, idx2)]),
        native_174_rgbd=native(3, 1), native_174_five_channels=dict(native(3, 1, 1), k=8, cout=64),
        cout_64_k8_8ch=dict(srcs=[src(rgb, 3), src(depth, 3), src(goal, 1), src(p(), 1)], cout=64, k=8, stride=1),
        k1_s1_1ch=dict(srcs=[src(depth, 1)], k=1, stride=1, cout=8),
        n0=dict(srcs=[src(rgb, 3, n=0), src(depth, 1, n=0)]),
        n0_store=dict(srcs=[dict(store(rgb, 3, idx), n=0), dict(store(depth, 1, idx), n=0)]),
        f16=dict(dtype=F16), odd_pixels=dict(cout=8, k=3, stride=2),   # 41 x 41
        dtype_zero=dict(dtype=0), dtype_three=dict(dtype=3), dtype_minus_one=dict(dtype=-1))
    E = {}

    def forward(a):
        return lib.vn_conv_u8_planes_forward(frames(a), len(a["srcs"]), a["weight"], a["bias"], a["cout"], a["k"],
                                             a["stride"], a["out"], None)

    def forward_lp(a):
        return lib.vn_conv_u8_planes_forward_lp(frames(a), len(a["srcs"]), a["weight"], a["bias"], a["cout"], a["k"],
                                                a["stride"], a["dtype"], a["out"], None)

    fa = dict(accepted, weight=p(), bias=p(), out=p())
    fwd_cases = dict(cases, null_weight=dict(weight=None), null_out=dict(out=None), no_bias=dict(bias=None),
                     off2_weight=dict(weight=fa["weight"] + 2), off2_bias=dict(bias=fa["bias"] + 2),
                     off2_out=dict(out=fa["out"] + 2), off1_out=dict(out=fa["out"] + 1))

    def need(a):
        c = max(sum(s["c"] for s in a["srcs"]), 1)
        n = max(a["srcs"][0]["n"], 0) if a["srcs"] else 0
        return lib.vn_conv_u8_wgrad_scratch_bytes(n, c, max(a["cout"], 1), max(a["k"], 1))

    def backward(a):
        return lib.vn_conv_u8_planes_backward(frames(a), len(a["srcs"]), a["grad_out"], a["cout"], a["k"], a["stride"],
                                              a["grad_weight"], a["grad_bias"], a["scratch"],
                                              need(a) + a["scratch_delta"], None)

    def backward_lp(a):
        return lib.vn_conv_u8_planes_backward_lp(frames(a), len(a["srcs"]), a["grad_out"], a["dtype"], a["cout"],
                                                 a["k"], a["stride"], a["grad_weight"], a["grad_bias"], a["scratch"],
                                                 need(a) + a["scratch_delta"], None)

    ba = dict(accepted, grad_out=p(), grad_weight=p(), grad_bias=p(), scratch=p(), scratch_delta=0)
    bwd_cases = dict(cases, null_grad_out=dict(grad_out=None), null_grad_weight=dict(grad_weight=None),
                     no_grad_bias=dict(grad_bias=None), null_scratch=dict(scratch=None),
                     scratch_off8=dict(scratch=ba["scratch"] + 8), scratch_short=dict(scratch_delta=-4),
                     n0_no_scratch=dict(cases["n0"], scratch=None), off2_grad_out=dict(grad_out=ba["grad_out"] + 2),
                     off1_grad_out=dict(grad_out=ba["grad_out"] + 1),
                     off2_grad_weight=dict(grad_weight=ba["grad_weight"] + 2),
                     off2_grad_bias=dict(grad_bias=ba["grad_bias"] + 2))
    for name, fn, a, cs in (("vn_conv_u8_planes_forward", forward, fa, fwd_cases),
                            ("vn_conv_u8_planes_forward_lp", forward_lp, fa, fwd_cases),
                            ("vn_conv_u8_planes_backward", backward, ba, bwd_cases),
                            ("vn_conv_u8_planes_backward_lp", backward_lp, ba, bwd_cases)):
        wanted = set(EXPECTED[name]) | set(_ACCEPTED) | set(_EXTRA_OK[name].split())
        E[name] = (fn, a, {k: v for k, v in cs.items() if k in wanted})
    return lib, E, keep


def arg_check_table():
    """{"entry point/case": [return code, the message it left or None when it left none of its own]}, plus the scratch
    sizes of a few plane sets."""
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    lib, E, _keep = _entry_points(vn)
    table = {}
    for name, (fn, accepted, cases) in E.items():
        for case, changed in [("accepted", {})] + sorted(cases.items()):
            lib.vn_gather_plane(None, 0, None, 0, None, 0, None)   # leaves the message "store: null"
            sentinel = lib.vn_last_error()
            rc = fn(dict(accepted, **changed))
            msg = lib.vn_last_error()
            table["%s/%s" % (name, case)] = [rc, msg.decode() if msg and msg != sentinel else None]
    sizes = {"%d,%d,%d,%d" % args: lib.vn_conv_u8_wgrad_scratch_bytes(*args)
             for args in ((81920, 4, 32, 7), (81920, 6, 32, 7), (8192, 8, 64, 8), (1, 5, 64, 8))}
    return dict(table=table, scratch=sizes)


def test_conv_u8_planes_argument_checks():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_conv_u8_planes_arg_checks as t; "
            "print(json.dumps(t.arg_check_table()))" % (ROOT, os.path.join(ROOT, "tests")))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr
    out = json.loads(res.stdout.strip().splitlines()[-1])
    seen = set()
    for key, (rc, msg) in out["table"].items():
        name, case = key.split("/")
        seen.add(key)
        if case in EXPECTED[name]:
            want_rc, want_msg = EXPECTED[name][case]
            assert rc == want_rc, (key, rc, msg)
            assert msg is not None and msg.startswith(name[3:] + ": ") and want_msg in msg, (key, msg)
        elif case in _ACCEPTED and _ACCEPTED[case] == OK or case == "n0_no_scratch":
            assert rc == OK, (key, rc, msg)
        else:   # passed validation: fails at the first CUDA call in a process without a device
            assert rc == ECUDA, (key, rc, msg)
    for name, cases in EXPECTED.items():
        missing = {"%s/%s" % (name, c) for c in list(cases) + list(_ACCEPTED) + _EXTRA_OK[name].split()} - seen
        assert not missing, missing
    for args, nbytes in out["scratch"].items():
        n, c, cout, k = map(int, args.split(","))
        assert nbytes == (n + 31) // 32 * cout * (c * k * k + 1) * 4, (args, nbytes)
