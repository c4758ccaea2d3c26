"""Which arguments the 16-bit (autocast) entry points of the uint8-frame convolution accept and which they reject, and the
return code of each.  As in test_conv_u8_arg_checks.py, a process that sees no CUDA device runs every call: the
descriptors carry aligned addresses that are never dereferenced, and a call that passes validation fails at its first
CUDA runtime call with VN_ECUDA.  Every case differs from the accepted call of its entry point in one argument.

The alignment rule pinned here: out and grad_out (16-bit) must be 2-byte aligned, so any oh * ow works, odd ones
included; weight, bias, grad_weight and grad_bias (fp32) 4-byte aligned; scratch 16-byte aligned."""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import test_conv_u8_arg_checks as fp32_checks  # noqa: E402

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, -1, -2, -3
F16, BF16 = 1, 2
_SHARED = fp32_checks._SHARED
_DTYPES = "dtype_minus_one dtype_three dtype_zero dtype_zero_n0"
EXPECTED = {
    "vn_conv_u8_forward_lp": {
        OK: "n0 n0_store",
        EINVAL: _SHARED["EINVAL"] + " null_out null_weight off1_out off2_bias off2_weight",
        ECUDA: "accepted cout_64_k8 depth f16 native_174 no_bias odd_pixels off2_out store_indices",
        EUNSUPPORTED: _SHARED["EUNSUPPORTED"] + " " + _DTYPES,
    },
    "vn_conv_u8_backward_lp": {
        OK: "n0 n0_no_scratch n0_store",
        EINVAL: _SHARED["EINVAL"] + (" null_grad_out null_grad_weight null_scratch off1_grad_out off2_grad_bias "
                                     "off2_grad_weight scratch_off8 scratch_short"),
        ECUDA: "accepted cout_64_k8 depth f16 native_174 no_grad_bias odd_pixels off2_grad_out store_indices",
        EUNSUPPORTED: _SHARED["EUNSUPPORTED"] + " " + _DTYPES,
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
               cout=32, k=7, stride=4, dtype=BF16)
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
        cout_64_k8=dict(cout=64, k=8), f16=dict(dtype=F16), odd_pixels=dict(cout=8, k=3, stride=2),   # 41 x 41
        dtype_zero=dict(dtype=0), dtype_three=dict(dtype=3), dtype_minus_one=dict(dtype=-1),
        dtype_zero_n0=dict(dtype=0, n=0))
    E = {}

    def forward(a):
        return lib.vn_conv_u8_forward_lp(frames(a), a["weight"], a["bias"], a["cout"], a["k"], a["stride"], a["dtype"],
                                         a["out"], None)

    a = dict(src, weight=p(), bias=p(), out=p())
    E["vn_conv_u8_forward_lp"] = (forward, a, dict(
        common, null_weight=dict(weight=None), null_out=dict(out=None), no_bias=dict(bias=None),
        off2_weight=dict(weight=a["weight"] + 2), off2_bias=dict(bias=a["bias"] + 2), off1_out=dict(out=a["out"] + 1),
        off2_out=dict(out=a["out"] + 2)))

    def backward(a):
        need = lib.vn_conv_u8_wgrad_scratch_bytes(max(a["n"], 0), max(a["c"], 1), max(a["cout"], 1), max(a["k"], 1))
        return lib.vn_conv_u8_backward_lp(frames(a), a["grad_out"], a["dtype"], a["cout"], a["k"], a["stride"],
                                          a["grad_weight"], a["grad_bias"], a["scratch"], need + a["scratch_delta"],
                                          None)

    a = dict(src, grad_out=p(), grad_weight=p(), grad_bias=p(), scratch=p(), scratch_delta=0)
    E["vn_conv_u8_backward_lp"] = (backward, a, dict(
        common, null_grad_out=dict(grad_out=None), null_grad_weight=dict(grad_weight=None),
        no_grad_bias=dict(grad_bias=None), null_scratch=dict(scratch=None), scratch_off8=dict(scratch=a["scratch"] + 8),
        scratch_short=dict(scratch_delta=-4), n0_no_scratch=dict(n=0, scratch=None),
        off1_grad_out=dict(grad_out=a["grad_out"] + 1), off2_grad_out=dict(grad_out=a["grad_out"] + 2),
        off2_grad_weight=dict(grad_weight=a["grad_weight"] + 2), off2_grad_bias=dict(grad_bias=a["grad_bias"] + 2)))
    return lib, E, keep


def arg_check_table():
    """{"entry point/case": [return code, whether a rejected call left a message of its own]}."""
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
    return dict(table=table)


def test_conv_u8_lp_argument_checks():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_conv_u8_lp_arg_checks as t; "
            "print(json.dumps(t.arg_check_table()))" % (os.path.dirname(ROOT), ROOT))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", code], cwd=os.path.dirname(ROOT), env=env,
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    got = {}
    for key, (rc, has_message) in json.loads(res.stdout.strip().splitlines()[-1])["table"].items():
        name, case = key.split("/")
        got.setdefault(name, {}).setdefault(rc, set()).add(case)
        assert has_message, "%s was rejected without a message of its own" % key
    assert got == {name: {rc: set(cases.split()) for rc, cases in by_rc.items()} for name, by_rc in EXPECTED.items()}
