"""Which arguments the uint8-frame convolution (vn_conv.cu) accepts and which it rejects, and the return code of each.
As in test_rollout_arg_checks.py, a process that sees no CUDA device runs every call: the descriptors carry aligned
addresses that are never dereferenced, and a call that passes validation fails at its first CUDA runtime call (the
shared-memory attribute) with VN_ECUDA.  Every case differs from the accepted call of its entry point in one argument.
Also pins sizeof(vn_u8_frames_t) and the weight-gradient scratch formula."""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, -1, -2, -3

_SHARED = dict(
    EINVAL=("base_null base_off8 h_zero idx_t_not_dividing_n idx_t_zero n_negative pitch_below_frame "
            "pitch_not_multiple_of_16 src_null"),
    EUNSUPPORTED=("channels_two cout_12 cout_72 frame_175 frame_below_kernel kernel_9 kernel_zero stride_above_kernel "
                  "stride_zero unsupported_n0"),
)
EXPECTED = {
    "vn_conv_u8_forward": {
        OK: "n0 n0_store",
        EINVAL: _SHARED["EINVAL"] + " null_out null_weight off2_bias off2_out off2_weight",
        ECUDA: "accepted cout_64_k8 depth native_174 no_bias store_indices",
        EUNSUPPORTED: _SHARED["EUNSUPPORTED"],
    },
    "vn_conv_u8_backward": {
        OK: "n0 n0_no_scratch n0_store",
        EINVAL: _SHARED["EINVAL"] + (" null_grad_out null_grad_weight null_scratch off2_grad_bias off2_grad_out "
                                     "off2_grad_weight scratch_off8 scratch_short"),
        ECUDA: "accepted cout_64_k8 depth native_174 no_grad_bias store_indices",
        EUNSUPPORTED: _SHARED["EUNSUPPORTED"],
    },
}


def _entry_points(vn):
    L = vn.lib
    lib = L.load()
    addr = iter(range(2 << 32, 3 << 32, 1 << 24))

    def p():
        return next(addr)

    keep = []

    def frames(a):
        f = L.U8Frames(a["base"], a["pitch"], a["idx"], a["sn"], a["st"], a["n"], a["idx_t"], a["h"], a["w"], a["c"], 0)
        keep.append(f)
        return None if a["null_src"] else C.byref(f)

    src = dict(null_src=False, base=p(), pitch=84 * 84 * 3, idx=None, sn=0, st=0, n=16, idx_t=1, h=84, w=84, c=3,
               cout=32, k=7, stride=4)
    common = dict(
        src_null=dict(null_src=True), base_null=dict(base=None), base_off8=dict(base=src["base"] + 8),
        pitch_not_multiple_of_16=dict(pitch=84 * 84 * 3 + 8), pitch_below_frame=dict(pitch=84 * 84 * 3 - 16),
        n_negative=dict(n=-1), h_zero=dict(h=0), n0=dict(n=0), n0_store=dict(n=0, idx=p(), pitch=100352, idx_t=4),
        idx_t_zero=dict(idx=p(), idx_t=0), idx_t_not_dividing_n=dict(idx=p(), idx_t=5),
        store_indices=dict(idx=p(), pitch=100352, idx_t=4, sn=1, st=4),
        channels_two=dict(c=2, pitch=84 * 84 * 3), kernel_zero=dict(k=0, stride=0), kernel_9=dict(k=9),
        stride_zero=dict(stride=0), stride_above_kernel=dict(k=3, stride=4), cout_12=dict(cout=12),
        cout_72=dict(cout=72), frame_175=dict(h=175, w=175, pitch=175 * 175 * 3 + 13),
        frame_below_kernel=dict(h=6, w=6, pitch=112), unsupported_n0=dict(cout=12, n=0),
        depth=dict(c=1, pitch=84 * 84), native_174=dict(h=174, w=174, pitch=90832),
        cout_64_k8=dict(cout=64, k=8))
    E = {}

    def forward(a):
        return lib.vn_conv_u8_forward(frames(a), a["weight"], a["bias"], a["cout"], a["k"], a["stride"], a["out"], None)

    a = dict(src, weight=p(), bias=p(), out=p())
    E["vn_conv_u8_forward"] = (forward, a, dict(
        common, null_weight=dict(weight=None), null_out=dict(out=None), no_bias=dict(bias=None),
        off2_weight=dict(weight=a["weight"] + 2), off2_bias=dict(bias=a["bias"] + 2), off2_out=dict(out=a["out"] + 2)))

    def backward(a):
        need = lib.vn_conv_u8_wgrad_scratch_bytes(max(a["n"], 0), max(a["c"], 1), max(a["cout"], 1), max(a["k"], 1))
        return lib.vn_conv_u8_backward(frames(a), a["grad_out"], a["cout"], a["k"], a["stride"], a["grad_weight"],
                                       a["grad_bias"], a["scratch"], need + a["scratch_delta"], None)

    a = dict(src, grad_out=p(), grad_weight=p(), grad_bias=p(), scratch=p(), scratch_delta=0)
    E["vn_conv_u8_backward"] = (backward, a, dict(
        common, null_grad_out=dict(grad_out=None), null_grad_weight=dict(grad_weight=None),
        no_grad_bias=dict(grad_bias=None), null_scratch=dict(scratch=None), scratch_off8=dict(scratch=a["scratch"] + 8),
        scratch_short=dict(scratch_delta=-4), n0_no_scratch=dict(n=0, scratch=None),
        off2_grad_out=dict(grad_out=a["grad_out"] + 2), off2_grad_weight=dict(grad_weight=a["grad_weight"] + 2),
        off2_grad_bias=dict(grad_bias=a["grad_bias"] + 2)))
    return lib, E, keep


def arg_check_table():
    """{"entry point/case": [return code, whether a rejected call left a message of its own]}, plus the struct size and
    a few scratch sizes."""
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    lib, E, _keep = _entry_points(vn)
    table = {}
    for name, (fn, accepted, cases) in E.items():
        for case, changed in [("accepted", {})] + sorted(cases.items()):
            lib.vn_gather_plane(None, 0, None, 0, None, 0, None)   # leaves the message "store: null"
            sentinel = lib.vn_last_error()
            rc = fn(dict(accepted, **changed))
            msg = lib.vn_last_error()
            table["%s/%s" % (name, case)] = [rc, rc == OK or (bool(msg) and msg != sentinel)]
    sizes = {"%d,%d,%d,%d" % args: lib.vn_conv_u8_wgrad_scratch_bytes(*args)
             for args in ((0, 3, 32, 7), (1, 3, 32, 7), (32, 3, 32, 7), (33, 3, 32, 7), (81920, 3, 32, 7),
                          (8192, 1, 16, 8), (-1, 3, 32, 7), (5, 3, 0, 7))}
    return dict(table=table, struct_size=lib.vn_abi_struct_size(9), sizeof_mirror=C.sizeof(vn.lib.U8Frames),
                scratch=sizes)


def _check(res):
    got = {}
    for key, (rc, has_message) in res["table"].items():
        name, case = key.split("/")
        got.setdefault(name, {}).setdefault(rc, set()).add(case)
        assert has_message, "%s was rejected without a message of its own" % key
    assert got == {name: {rc: set(cases.split()) for rc, cases in by_rc.items()} for name, by_rc in EXPECTED.items()}
    assert res["struct_size"] == res["sizeof_mirror"] == 64
    chunks = lambda n: (n + 31) // 32
    for args, nbytes in res["scratch"].items():
        n, c, cout, k = map(int, args.split(","))
        want = -1 if n < 0 or cout < 1 else chunks(n) * cout * (c * k * k + 1) * 4
        assert nbytes == want, (args, nbytes, want)


def test_conv_u8_argument_checks():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_conv_u8_arg_checks as t; "
            "print(json.dumps(t.arg_check_table()))" % (ROOT, os.path.join(ROOT, "tests")))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr
    _check(json.loads(res.stdout.strip().splitlines()[-1]))
