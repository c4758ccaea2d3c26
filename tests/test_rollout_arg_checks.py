"""Which arguments the rollout builders (every entry point of vn_rollout.cu) accept and which they reject, and the
return code of each.  A process that sees no CUDA device runs every call: the descriptors carry aligned addresses that
are never dereferenced, and a call that passes validation fails at its first CUDA runtime call (the shared-memory
attribute or the launch) with VN_ECUDA, so nothing reaches a GPU and the table is the same with or without one.
Every case differs from the accepted call of its entry point in one argument."""
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (h, w, c) of the planes of the fake store: RGB, depth, a 2-channel plane, a frame too large for shared memory, a frame
# of which one copy fits shared memory but two do not, and a frame whose pixel count is not a multiple of 4
PLANES = ((84, 84, 3), (84, 84, 1), (84, 84, 2), (300, 300, 3), (200, 200, 3), (83, 83, 1))
RGB, DEPTH, TWO_CH, HUGE, BIG, ODD = range(len(PLANES))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, -1, -2, -3

# Return code -> cases, per entry point.  ECUDA marks a call that passed validation.
EXPECTED = {
    "vn_gather_plane_f32_chw": {
        OK: "huge_frame_staged_n0 n0",
        EINVAL: (
            "huge_frame_staged n_negative null_idx null_out plane_bytes_mismatch plane_negative plane_past_end "
            "store_base_null store_null store_pitch_unaligned store_plane_off_unaligned"
        ),
        ECUDA: "accepted huge_frame_vectorised odd_pixels_staged staged_out_off4 two_channels_staged",
    },
    "vn_gather_plane_f32_chw_rows": {
        OK: "huge_frame_staged_n0 n0",
        EINVAL: (
            "huge_frame_staged idx_stride_zero n_negative null_idx null_out plane_bytes_mismatch plane_negative "
            "plane_past_end store_base_null store_null store_pitch_unaligned store_plane_off_unaligned"
        ),
        ECUDA: "accepted huge_frame_vectorised odd_pixels_staged staged_out_off4 two_channels_staged",
    },
    "vn_gather_leaves_f32_chw": {
        OK: "n0",
        EINVAL: (
            "leaf_out_null leaf_out_off4 leaf_plane_bytes_mismatch leaf_plane_past_end leaf_source_two "
            "n_leaves_seven n_leaves_seven_n0 n_leaves_zero n_negative null_desc null_leaves store_base_null "
            "store_null store_pitch_unaligned store_plane_off_unaligned"
        ),
        ECUDA: "accepted huge_frame",
        EUNSUPPORTED: "odd_pixels odd_pixels_n0 two_channels two_channels_n0",
    },
    "vn_nstep_returns": {
        OK: "n0",
        EINVAL: "n_negative null_done null_last_value null_out null_reward t_zero",
        ECUDA: "accepted",
    },
    "vn_nstep_returns_scan": {
        OK: "n0",
        EINVAL: "n_negative null_done null_last_value null_out null_reward t_zero",
        ECUDA: "accepted",
    },
    "vn_discounted_backup": {
        OK: "n0",
        EINVAL: "d_zero n_negative null_bootstrap null_done null_out null_reward t_zero",
        ECUDA: "accepted",
    },
    "vn_pixel_control": {
        OK: "huge_frame_n0 n0 two_frames_too_large_n0",
        EINVAL: (
            "huge_frame n_negative null_out null_states plane_bytes_mismatch plane_negative plane_past_end "
            "pool_cell_zero pool_larger_than_frame pool_larger_than_frame_n0 pool_out_h_zero store_base_null "
            "store_null store_pitch_unaligned store_plane_off_unaligned t_zero two_frames_too_large"
        ),
        ECUDA: "accepted too_many_blocks",
    },
    "vn_transition_rows": {
        OK: "n0",
        EINVAL: "n_negative null_adj null_miss_count null_miss_pos null_rows null_states off4_adj t_zero",
        ECUDA: "accepted",
    },
    "vn_gather_rows": {
        OK: "n0 n_negative",
        EINVAL: (
            "idx_t_zero n_not_multiple_of_idx_t null_idx null_out null_table off4_out off4_table "
            "row_bytes_not_multiple_of_16 row_bytes_zero"
        ),
        ECUDA: "accepted",
    },
    "vn_pixel_control_list": {
        OK: "huge_frame_max_count_zero huge_frame_n0 max_count_zero n0",
        EINVAL: (
            "huge_frame max_count_negative n_negative null_count null_out null_pos null_states "
            "plane_bytes_mismatch plane_negative plane_past_end pool_cell_zero pool_larger_than_frame "
            "pool_larger_than_frame_n0 pool_out_h_zero store_base_null store_null store_pitch_unaligned "
            "store_plane_off_unaligned t_zero two_frames_too_large"
        ),
        ECUDA: "accepted compact",
    },
    "vn_pixel_control_returns": {
        OK: "n0",
        EINVAL: (
            "cells_not_multiple_of_4 cells_zero n_negative null_bootstrap null_done null_miss_rows "
            "null_out_returns null_pc_table null_rows off4_bootstrap off4_miss_rows off4_out_returns "
            "off4_out_reward off4_pc_table t_zero"
        ),
        ECUDA: "accepted no_out_reward",
    },
    "vn_pixel_control_returns_from_states": {
        OK: "huge_frame_n0 n0",
        EINVAL: (
            "cells_below_4 cells_not_multiple_of_4 max_miss_zero n_negative null_adj null_bootstrap null_done "
            "null_miss_count null_miss_pos null_miss_rows null_out_returns null_pc_table null_rows null_states "
            "off4_adj off4_bootstrap off4_miss_rows off4_out_returns off4_out_reward off4_pc_table "
            "plane_bytes_mismatch plane_negative plane_past_end pool_cell_zero pool_larger_than_frame "
            "pool_larger_than_frame_n0 pool_out_h_zero store_base_null store_null store_pitch_unaligned "
            "store_plane_off_unaligned t_zero"
        ),
        ECUDA: "accepted huge_frame no_out_reward two_frames_too_large",
    },
    "vn_replay_sample": {
        OK: "n0",
        EINVAL: (
            "cap_zero count_negative count_past_cap head_negative head_past_end length_zero mode_two n_negative "
            "null_o_actions null_o_dones null_o_goals null_o_rewards null_o_start null_o_states null_ring "
            "null_ring_action null_ring_after null_ring_before null_ring_done null_ring_goal "
            "null_ring_goal_before null_ring_reward"
        ),
        ECUDA: "accepted length_zero_rp_mode rp_mode_with_label",
    },
    "vn_aux_target": {
        OK: "huge_frame_n0 n0",
        EINVAL: (
            "huge_frame n_negative null_idx null_out plane_bytes_mismatch plane_negative plane_past_end "
            "pool_cell_zero pool_larger_than_frame pool_larger_than_frame_m0 pool_out_h_zero store_base_null "
            "store_null store_pitch_unaligned store_plane_off_unaligned"
        ),
        ECUDA: "accepted big_frame",
    },
    "vn_rp_labels": {
        OK: "n0",
        EINVAL: "n_negative n_not_multiple_of_t n_past_2_24 null_reward null_scratch t_zero",
        ECUDA: "accepted many_blocks n_at_2_24 no_labels no_lists",
    },
}


def _entry_points(vn):
    """{entry point: (call, accepted arguments, {case: changed arguments})}"""
    L = vn.lib
    lib = L.load()
    addr = iter(range(2 << 32, 3 << 32, 1 << 24))   # distinct, 16-byte aligned; nothing is read or written there

    def p():
        return next(addr)

    def store(pitch_delta=0, off0=0, base=1 << 32):
        s = L.Store()
        s.base = base
        s.n_states = 6000
        s.n_planes = len(PLANES)
        off = 0
        for i, (h, w, c) in enumerate(PLANES):
            s.plane_off[i] = off + off0
            s.plane_bytes[i] = (h * w * c + 15) & ~15
            off = (off + s.plane_bytes[i] + 127) & ~127
        s.state_pitch = off + pitch_delta
        return s

    good = store()
    stores = dict(good=C.byref(good), null=None, null_base=C.byref(store(base=0)),
                  pitch4=C.byref(store(pitch_delta=4)), off8=C.byref(store(off0=8)))
    keep = [good, stores]

    def frame(plane, pool=True):
        h, w, c = PLANES[plane]
        a = dict(plane=plane, h=h, w=w, c=c)
        if pool:
            a.update(cell=4, out_h=20, out_w=20)
        return a

    def store_cases(a):
        """The store / plane / geometry cases of an entry point that reads frames."""
        return {"store_null": dict(store="null"), "store_base_null": dict(store="null_base"),
                "store_pitch_unaligned": dict(store="pitch4"), "store_plane_off_unaligned": dict(store="off8"),
                "plane_negative": dict(plane=-1), "plane_past_end": dict(plane=len(PLANES)),
                "plane_bytes_mismatch": dict(h=a["h"] - 4)}

    def pool_cases():
        return {"pool_cell_zero": dict(cell=0), "pool_out_h_zero": dict(out_h=0),
                "pool_larger_than_frame": dict(out_h=22, out_w=22), "pool_larger_than_frame_n0": dict(out_h=22, out_w=22, n=0)}

    def nulls(a, *names):
        return {"null_" + k: {k: None} for k in names}

    def off4(a, *names):
        return {"off4_" + k: {k: a[k] + 4} for k in names}

    E = {}

    def gather_rows_f32(a):
        return lib.vn_gather_plane_f32_chw_rows(stores[a["store"]], a["plane"], a["idx"], a["idx_stride"], a["n"], a["h"],
                                                a["w"], a["c"], a["out"], None)

    def gather_f32(a):
        return lib.vn_gather_plane_f32_chw(stores[a["store"]], a["plane"], a["idx"], a["n"], a["h"], a["w"], a["c"],
                                           a["out"], None)

    for name, fn, strided in (("vn_gather_plane_f32_chw", gather_f32, False),
                              ("vn_gather_plane_f32_chw_rows", gather_rows_f32, True)):
        a = dict(store="good", idx=p(), idx_stride=2 if strided else 1, n=8, out=p(), **frame(RGB, False))
        cases = dict(store_cases(a), **nulls(a, "idx", "out"))
        cases.update(n0=dict(n=0), n_negative=dict(n=-1),
                     staged_out_off4=dict(out=a["out"] + 4),
                     two_channels_staged=frame(TWO_CH, False),
                     huge_frame_vectorised=frame(HUGE, False),
                     huge_frame_staged=dict(frame(HUGE, False), out=a["out"] + 4),
                     huge_frame_staged_n0=dict(frame(HUGE, False), out=a["out"] + 4, n=0),
                     odd_pixels_staged=frame(ODD, False))
        if strided:
            cases.update(idx_stride_zero=dict(idx_stride=0))
        E[name] = (fn, a, cases)

    def leaves(a):
        arr = (L.FloatLeaf * len(a["leaves"]))()
        for i, (plane, source, channels, out) in enumerate(a["leaves"]):
            arr[i].plane, arr[i].source, arr[i].channels, arr[i].out = plane, source, channels, out
        keep.append(arr)
        return lib.vn_gather_leaves_f32_chw(stores[a["store"]], None if a["null_leaves"] else arr, a["n_leaves"],
                                            a["desc"], a["n"], a["h"], a["w"], None)

    lv = [(RGB, 0, 3, p()), (DEPTH, 1, 1, p())]

    def leaf(i, **kw):
        t = dict(zip(("plane", "source", "channels", "out"), lv[i]), **kw)
        return [tuple(t[k] for k in ("plane", "source", "channels", "out")) if j == i else lv[j] for j in range(len(lv))]

    a = dict(store="good", leaves=lv, null_leaves=False, n_leaves=2, desc=p(), n=8, h=84, w=84)
    E["vn_gather_leaves_f32_chw"] = (leaves, a, dict(
        n0=dict(n=0), n_negative=dict(n=-1), store_null=dict(store="null"), store_base_null=dict(store="null_base"),
        store_pitch_unaligned=dict(store="pitch4"), store_plane_off_unaligned=dict(store="off8"),
        null_leaves=dict(null_leaves=True), null_desc=dict(desc=None),
        n_leaves_zero=dict(n_leaves=0), n_leaves_seven=dict(n_leaves=7, leaves=lv * 4),
        n_leaves_seven_n0=dict(n_leaves=7, leaves=lv * 4, n=0),
        odd_pixels=dict(h=83, w=83, leaves=[(ODD, 0, 1, lv[0][3])], n_leaves=1),
        odd_pixels_n0=dict(h=83, w=83, leaves=[(ODD, 0, 1, lv[0][3])], n_leaves=1, n=0),
        two_channels=dict(leaves=leaf(0, plane=TWO_CH, channels=2)),
        two_channels_n0=dict(leaves=leaf(0, plane=TWO_CH, channels=2), n=0),
        leaf_plane_past_end=dict(leaves=leaf(1, plane=len(PLANES))),
        leaf_plane_bytes_mismatch=dict(leaves=leaf(0, channels=1)),
        leaf_out_null=dict(leaves=leaf(1, out=None)), leaf_out_off4=dict(leaves=leaf(1, out=lv[1][3] + 4)),
        leaf_source_two=dict(leaves=leaf(1, source=2)), huge_frame=dict(h=300, w=300, leaves=[(HUGE, 0, 3, p())],
                                                                       n_leaves=1)))

    for name in ("vn_nstep_returns", "vn_nstep_returns_scan"):
        fn = getattr(lib, name)
        a = dict(reward=p(), done=p(), last_value=p(), out=p(), n=4, t=5)
        E[name] = ((lambda a, fn=fn: fn(a["reward"], a["done"], a["last_value"], 0.99, a["n"], a["t"], 1, a["n"],
                                        a["out"], a["t"], 1, None)), a,
                   dict(nulls(a, "reward", "done", "last_value", "out"), n0=dict(n=0), n_negative=dict(n=-1),
                        t_zero=dict(t=0)))

    a = dict(reward=p(), done=p(), bootstrap=p(), out=p(), n=4, t=5, d=400)
    E["vn_discounted_backup"] = (
        lambda a: lib.vn_discounted_backup(a["reward"], a["done"], a["t"], 1, a["bootstrap"], 0.9, a["n"], a["t"], a["d"],
                                           a["out"], None), a,
        dict(nulls(a, "reward", "done", "bootstrap", "out"), n0=dict(n=0), n_negative=dict(n=-1), t_zero=dict(t=0),
             d_zero=dict(d=0)))

    a = dict(store="good", states=p(), n=4, t=5, out=p(), **frame(RGB))
    E["vn_pixel_control"] = (
        lambda a: lib.vn_pixel_control(stores[a["store"]], a["plane"], a["states"], a["n"], a["t"], a["t"] + 1, 1, a["h"],
                                       a["w"], a["c"], a["cell"], a["out_h"], a["out_w"], a["out"], None), a,
        dict(store_cases(a), **pool_cases(), **nulls(a, "states", "out"), n0=dict(n=0), n_negative=dict(n=-1),
             t_zero=dict(t=0), huge_frame=frame(HUGE), huge_frame_n0=dict(frame(HUGE), n=0),
             two_frames_too_large=frame(BIG), two_frames_too_large_n0=dict(frame(BIG), n=0),
             too_many_blocks=dict(n=(1 << 31) - 1, t=17)))

    a = dict(adj=p(), states=p(), n=4, t=5, rows=p(), miss_pos=p(), miss_count=p())
    E["vn_transition_rows"] = (
        lambda a: lib.vn_transition_rows(a["adj"], a["states"], a["n"], a["t"], 1, a["n"], a["rows"], a["t"], 1,
                                         a["miss_pos"], a["miss_count"], None), a,
        dict(nulls(a, "adj", "states", "rows", "miss_pos", "miss_count"), **off4(a, "adj"), n0=dict(n=0),
             n_negative=dict(n=-1), t_zero=dict(t=0)))

    a = dict(table=p(), row_bytes=1600, idx=p(), n=20, idx_t=5, out=p())
    E["vn_gather_rows"] = (
        lambda a: lib.vn_gather_rows(a["table"], a["row_bytes"], a["idx"], a["n"], a["idx_t"], 1, a["n"] // 5, a["out"],
                                     None), a,
        dict(nulls(a, "table", "idx", "out"), **off4(a, "table", "out"), n0=dict(n=0), n_negative=dict(n=-5),
             idx_t_zero=dict(idx_t=0), n_not_multiple_of_idx_t=dict(n=21), row_bytes_zero=dict(row_bytes=0),
             row_bytes_not_multiple_of_16=dict(row_bytes=1604)))

    a = dict(store="good", states=p(), n=4, t=5, pos=p(), count=p(), max_count=20, compact=0, out=p(), **frame(RGB))
    E["vn_pixel_control_list"] = (
        lambda a: lib.vn_pixel_control_list(stores[a["store"]], a["plane"], a["states"], a["n"], a["t"], 1, a["n"], a["h"],
                                            a["w"], a["c"], a["cell"], a["out_h"], a["out_w"], a["pos"], a["count"],
                                            a["max_count"], a["compact"], a["out"], None), a,
        dict(store_cases(a), **pool_cases(), **nulls(a, "states", "pos", "count", "out"), n0=dict(n=0),
             n_negative=dict(n=-1), t_zero=dict(t=0), max_count_zero=dict(max_count=0),
             max_count_negative=dict(max_count=-1), compact=dict(compact=1), huge_frame=frame(HUGE),
             huge_frame_n0=dict(frame(HUGE), n=0), huge_frame_max_count_zero=dict(frame(HUGE), max_count=0),
             two_frames_too_large=frame(BIG)))

    a = dict(pc_table=p(), cells=400, rows=p(), miss_rows=p(), done=p(), bootstrap=p(), n=4, t=5, out_returns=p(),
             out_reward=p())
    E["vn_pixel_control_returns"] = (
        lambda a: lib.vn_pixel_control_returns(a["pc_table"], a["cells"], a["rows"], a["t"], 1, a["miss_rows"], a["done"],
                                               1, a["n"], a["bootstrap"], 0.9, a["n"], a["t"], a["out_returns"],
                                               a["out_reward"], None), a,
        dict(nulls(a, "pc_table", "rows", "miss_rows", "done", "bootstrap", "out_returns"),
             **off4(a, "pc_table", "miss_rows", "bootstrap", "out_returns", "out_reward"), no_out_reward=dict(out_reward=None),
             n0=dict(n=0), n_negative=dict(n=-1), t_zero=dict(t=0), cells_zero=dict(cells=0),
             cells_not_multiple_of_4=dict(cells=402)))

    a = dict(store="good", adj=p(), pc_table=p(), states=p(), done=p(), bootstrap=p(), n=4, t=5, rows=p(), miss_pos=p(),
             miss_count=p(), miss_rows=p(), max_miss=20, out_returns=p(), out_reward=p(), **frame(RGB))
    E["vn_pixel_control_returns_from_states"] = (
        lambda a: lib.vn_pixel_control_returns_from_states(
            stores[a["store"]], a["plane"], a["adj"], a["pc_table"], a["states"], 1, a["n"], a["done"], 1, a["n"],
            a["bootstrap"], 0.9, a["n"], a["t"], a["h"], a["w"], a["c"], a["cell"], a["out_h"], a["out_w"], a["rows"],
            a["miss_pos"], a["miss_count"], a["miss_rows"], a["max_miss"], a["out_returns"], a["out_reward"], None), a,
        dict(store_cases(a), **pool_cases(),
             **nulls(a, "adj", "pc_table", "states", "done", "bootstrap", "rows", "miss_pos", "miss_count", "miss_rows",
                     "out_returns"),
             **off4(a, "adj", "pc_table", "miss_rows", "bootstrap", "out_returns", "out_reward"),
             no_out_reward=dict(out_reward=None), n0=dict(n=0), n_negative=dict(n=-1), t_zero=dict(t=0),
             max_miss_zero=dict(max_miss=0), cells_not_multiple_of_4=dict(out_h=19, out_w=19),
             cells_below_4=dict(out_h=1, out_w=2), huge_frame=frame(HUGE), huge_frame_n0=dict(frame(HUGE), n=0),
             two_frames_too_large=frame(BIG)))

    def replay(a):
        ring = L.Replay(*a["ring"])
        keep.append(ring)
        return lib.vn_replay_sample(None if a["null_ring"] else C.byref(ring), a["length"], a["mode"], C.c_uint64(7), 3,
                                    0, a["o_states"], a["o_goals"], a["o_actions"], a["o_rewards"], a["o_dones"],
                                    a["o_start"], a["o_label"], None)

    ring = [p() for _ in range(7)] + [8, 50, 10, 30]   # before, after, goal, goal_before, action, reward, done; n, cap, head, count

    def ring_with(**kw):
        names = ("before", "after", "goal", "goal_before", "action", "reward", "done", "n", "cap", "head", "count")
        return [kw.get(k, v) for k, v in zip(names, ring)]

    a = dict(ring=ring, null_ring=False, length=5, mode=0, o_states=p(), o_goals=p(), o_actions=p(), o_rewards=p(),
             o_dones=p(), o_start=p(), o_label=None)
    E["vn_replay_sample"] = (replay, a, dict(
        {"null_ring_" + k: dict(ring=ring_with(**{k: None}))
         for k in ("before", "after", "goal", "goal_before", "action", "reward", "done")},
        **nulls(a, "o_states", "o_goals", "o_actions", "o_rewards", "o_dones", "o_start"),
        null_ring=dict(null_ring=True), n0=dict(ring=ring_with(n=0)), n_negative=dict(ring=ring_with(n=-1)),
        cap_zero=dict(ring=ring_with(cap=0, head=0, count=0)), count_negative=dict(ring=ring_with(count=-1)),
        count_past_cap=dict(ring=ring_with(count=51)), head_negative=dict(ring=ring_with(head=-1)),
        head_past_end=dict(ring=ring_with(head=50)), mode_two=dict(mode=2), length_zero=dict(length=0),
        length_zero_rp_mode=dict(length=0, mode=1), rp_mode_with_label=dict(mode=1, o_label=p())))

    a = dict(store="good", idx=p(), m=8, out=p(), **frame(DEPTH))
    E["vn_aux_target"] = (
        lambda a: lib.vn_aux_target(stores[a["store"]], a["plane"], a["idx"], a["m"], a["h"], a["w"], a["c"], a["cell"],
                                    a["out_h"], a["out_w"], a["out"], None), a,
        dict(store_cases(a), **dict((k.replace("_n0", "_m0"), dict((("m" if x == "n" else x), y) for x, y in v.items()))
                                    for k, v in pool_cases().items()),
             **nulls(a, "idx", "out"), n0=dict(m=0), n_negative=dict(m=-1), huge_frame=frame(HUGE),
             huge_frame_n0=dict(frame(HUGE), m=0), big_frame=frame(BIG)))

    a = dict(reward=p(), n=20, t=5, labels=p(), zero=p(), nonzero=p(), counts=p(), scratch=p())
    E["vn_rp_labels"] = (
        lambda a: lib.vn_rp_labels(a["reward"], a["n"], a["t"], 1, a["n"] // max(a["t"], 1), a["labels"], a["zero"],
                                   a["nonzero"], a["counts"], a["scratch"], None), a,
        dict(nulls(a, "reward", "scratch"), no_lists=dict(zero=None, nonzero=None), no_labels=dict(labels=None),
             n0=dict(n=0), n_negative=dict(n=-5), n_past_2_24=dict(n=(1 << 24) + 4), n_at_2_24=dict(n=1 << 24, t=4),
             n_not_multiple_of_t=dict(n=21), t_zero=dict(t=0), many_blocks=dict(n=300 * 1024, t=4)))
    return lib, E, keep


def arg_check_table():
    """{"entry point/case": [return code, whether a rejected call left a message of its own]}"""
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
    return table


def _check(table):
    got = {}
    for key, (rc, has_message) in table.items():
        name, case = key.split("/")
        got.setdefault(name, {}).setdefault(rc, set()).add(case)
        assert has_message, "%s was rejected without a message of its own" % key
    assert got == {name: {rc: set("".join(cases).split()) for rc, cases in by_rc.items()}
                   for name, by_rc in EXPECTED.items()}


def test_rollout_argument_checks():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_rollout_arg_checks as t; "
            "print(json.dumps(t.arg_check_table()))" % (ROOT, os.path.join(ROOT, "tests")))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr
    _check(json.loads(res.stdout.strip().splitlines()[-1]))
