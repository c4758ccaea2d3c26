"""Which launch mode vn_env_step / vn_env_reset pick, and how many host_seq words a host-facing step publishes, for
the batch sizes, layouts, flags and variants the library serves.  The answers come from host logic alone: the
descriptors carry aligned pointers that are never dereferenced, and no kernel is launched, so the test runs without a
GPU (the library then assumes the B200's 148 SMs).  The same table must come back when the process environment holds
values for variables that once tuned the step path: the library reads none."""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

B200_SMS = 148
SIZES = (16, 444, 445, 777, 1024, 4096, 4144, 4145, 8192)
VARIANTS = ("AUTO", "LDG", "BULK", "FUSED", "PERSISTENT")
# (store planes, frame size, observation planes, goal planes)
LAYOUTS = {
    "c2": (("rgb", "depth"), (84, 84), ("rgb", "depth"), ("rgb",)),
    "rgb": (("rgb",), (84, 84), ("rgb",), ()),
    "aux5": (("rgb", "depth", "segmentation"), (84, 84), ("rgb", "depth", "segmentation"), ("rgb", "segmentation")),
    "native174": (("rgb", "depth", "segmentation"), (174, 174), ("rgb", "depth", "segmentation"),
                  ("rgb", "segmentation")),
}
RETIRED_VARIABLES = {
    "VN_NO_PDL": "1", "VN_NO_WHOLE_RECORD": "1", "VN_BULK_SPLIT": "3", "VN_BULK_PER_SM": "1", "VN_BULK_GRID": "7",
    "VN_BULK_DYNAMIC": "0", "VN_BULK_GROUPS": "4", "VN_BULK_L2_HINTS": "0", "VN_BULK_TAIL_SPLIT": "4",
    "VN_BULK_TAIL_WAVES16": "8", "VN_NO_FUSED": "1", "VN_FUSED_PER_SM": "1", "VN_PERSISTENT": "2",
}

# Mode per batch size (one character per entry of SIZES): 0 scalar kernel + gather kernel, 1 fused launch,
# 2 persistent launch, E rejected.  The four strings of a (layout, variant) are for: serial steps of a device caller,
# serial steps of a host caller (out->host_pack), pipelined steps (VN_STEP_ACTIONS_READY) of a device caller, pipelined
# steps of a host caller.
EXPECTED = {
    ("c2", "AUTO"): ("112222200", "110000000", "112200000", "110000000"),
    ("c2", "LDG"): ("000000000", "000000000", "000000000", "000000000"),
    ("c2", "BULK"): ("000000000", "000000000", "000000000", "000000000"),
    ("c2", "FUSED"): ("111111111", "111111111", "111111111", "111111111"),
    ("c2", "PERSISTENT"): ("222222222", "222222222", "222222222", "222222222"),
    ("rgb", "AUTO"): ("111222220", "111000000", "111220000", "111000000"),
    ("rgb", "LDG"): ("000000000", "000000000", "000000000", "000000000"),
    ("rgb", "BULK"): ("000000000", "000000000", "000000000", "000000000"),
    ("rgb", "FUSED"): ("111111111", "111111111", "111111111", "111111111"),
    ("rgb", "PERSISTENT"): ("222222222", "222222222", "222222222", "222222222"),
    ("aux5", "AUTO"): ("122220000", "100000000", "120000000", "100000000"),
    ("aux5", "LDG"): ("000000000", "000000000", "000000000", "000000000"),
    ("aux5", "BULK"): ("000000000", "000000000", "000000000", "000000000"),
    ("aux5", "FUSED"): ("111111111", "111111111", "111111111", "111111111"),
    ("aux5", "PERSISTENT"): ("222222222", "222222222", "222222222", "222222222"),
    ("native174", "AUTO"): ("000000000", "000000000", "000000000", "000000000"),
    ("native174", "LDG"): ("000000000", "000000000", "000000000", "000000000"),
    ("native174", "BULK"): ("000000000", "000000000", "000000000", "000000000"),
    ("native174", "FUSED"): ("EEEEEEEEE", "EEEEEEEEE", "EEEEEEEEE", "EEEEEEEEE"),
    ("native174", "PERSISTENT"): ("EEEEEEEEE", "EEEEEEEEE", "EEEEEEEEE", "EEEEEEEEE"),
}


def _layout(vn, name):
    planes, hw, obs, goal = LAYOUTS[name]
    lay = vn.tables.StoreLayout.make(planes, hw)
    L = vn.lib
    store = L.Store()
    store.base = 1 << 32
    store.state_pitch = lay.state_pitch
    store.n_states = 6000
    store.n_planes = len(planes)
    for i in range(len(planes)):
        store.plane_off[i] = lay.plane_off[i]
        store.plane_bytes[i] = lay.plane_bytes[i]
    out = L.StepOut()
    # distinct, 16-byte aligned addresses; nothing is read or written through them
    addr = iter(range(2 << 32, 3 << 32, 1 << 24))
    for i, p in enumerate(planes):
        if p in obs:
            out.obs[i] = next(addr)
        if p in goal:
            out.goal_obs[i] = next(addr)
    for f in ("reward", "done", "did_reset", "obs_state", "stats", "gather_desc", "sched"):
        setattr(out, f, next(addr))
    return store, out


def policy_table():
    """{"layout/variant": [(modes, host_seq words) for each flag combination of EXPECTED]} over every batch size."""
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    L = vn.lib
    lib = L.load()
    table = {}
    for name in LAYOUTS:
        store, out = _layout(vn, name)
        for v in VARIANTS:
            variant = getattr(L, "GATHER_" + v)
            rows = []
            for ready in (False, True):
                for host in (False, True):
                    out.flags = L.STEP_ACTIONS_READY if ready else 0
                    out.host_pack = (4 << 32) if host else None
                    out.host_seq = (5 << 32) if host else None
                    modes, words = "", []
                    for n in SIZES:
                        envs = L.Envs()
                        envs.n_envs = n
                        m = lib.vn_env_step_mode(C.byref(store), C.byref(envs), C.byref(out), variant)
                        modes += "E" if m < 0 else str(m)
                        words.append(lib.vn_env_host_seq_words(C.byref(store), C.byref(envs), C.byref(out), variant))
                    rows.append((modes, words))
            table["%s/%s" % (name, v)] = rows
    return table


def expected_words(modes):
    """One word per block of the scalar half: one per 128 envs, one per env of a fused launch, one for the whole
    persistent grid; an error where the mode is rejected."""
    per = {"0": lambda n: -(-n // 128), "1": lambda n: n, "2": lambda n: 1, "E": lambda n: -1}
    return [per[m](n) for m, n in zip(modes, SIZES)]


@pytest.fixture(scope="module")
def b200_like():
    try:
        import torch
        if torch.cuda.is_available() and torch.cuda.get_device_properties(0).multi_processor_count != B200_SMS:
            pytest.skip("the recorded table is for a device with %d SMs" % B200_SMS)
    except ImportError:
        pass


def _check(table):
    assert {tuple(k.split("/")): tuple(m for m, _ in rows) for k, rows in table.items()} == EXPECTED
    for key, rows in table.items():
        for modes, words in rows:
            assert words == expected_words(modes), key


def test_launch_policy_table(b200_like):
    _check(policy_table())


def test_launch_policy_ignores_the_environment(b200_like):
    env = dict(os.environ, **RETIRED_VARIABLES)
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_launch_policy as t; "
            "print(json.dumps(t.policy_table()))" % (ROOT, os.path.join(ROOT, "tests")))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr
    _check(json.loads(res.stdout.strip().splitlines()[-1]))
