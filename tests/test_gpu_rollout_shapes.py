"""Every rollout / target-builder kernel and launch shape (vn_rollout.cu) against exact and float64 references.

vn_rollout.cu holds 22 kernel instantiations, and its host code caps the grid of most of them, so a large enough batch
makes a kernel loop over its work.  ``CASES`` names, for each launch shape, the branch it is there for and the one-line
derivation from the host code's constants (the grid caps ``sm_count() * {8, 16, 64}`` and ``ctas_per_sm(smem, 4)``,
``kChunk``, ``kAhead``, ``kRpBlock``, the ``blocks > 256`` scan switch, the leaves unroll and ``kMaxSmem``);
``test_case_table_branches`` recomputes those branches on the CPU for a B200 (148 SMs), and every GPU test recomputes
them from the device's own SM count before it runs.

Exact family.  Every builder except the warp-scan returns is written in the oracle's fp32 operation order
(oracle/rollout.py: ``__fadd_rn`` / ``__fdiv_rn`` in the same order, and ``u8_over_255`` is correctly rounded for all
256 byte values), so pixel control (direct, table and list paths), the fused pixel-control returns, aux targets,
``discounted_backup``, the serial returns and the float gathers are compared bit for bit, as are the integer outputs
(RP labels and lists, replay draws, gathered rows).  Where an oracle input would be large the device paths are compared
with each other in full and with the oracle on a seeded sample of rows.

Bound family.  The warp-scan returns re-associate the recurrence; they are checked against a float64 recurrence with
an error bound taken from the scan's operation count, and the bound is shown to reject three wrong answers."""
import ctypes as C
import importlib
import re
import zlib
from collections import namedtuple
from functools import lru_cache

import numpy as np
import pytest

from oracle import rollout as orl

vn = importlib.import_module("a2cat-vn-pytorch_b200")

B200_SMS = 148
# vn_rollout.cu's host constants, for the derivations in CASES
SMEM = 220 * 1024                   # kMaxSmem (and the 220 KB ctas_per_sm divides)
K_CHUNK, K_AHEAD, RP_BLOCK = 16, 4, 1024
RP_SCAN_BLOCKS = 256                # vn_rp_labels runs the scan kernel when blocks > 256
LEAF_UNROLL = (4, 2, 2, 1, 1, 1)    # launch_float_leaves: unroll by leaf count
PLANE_C = {"rgb": 3, "depth": 1, "segmentation": 3}


def _cdiv(a, b):
    return -(-a // b)


def _pad16(x):
    return (x + 15) // 16 * 16


def _ctas_per_sm(smem, cap):
    return max(1, min(SMEM // (smem + 1024), cap))


Case = namedtuple("Case", "id kind p claims why")


def _plan(case, sms):
    """What vn_rollout.cu's host code picks for `case` on a device with `sms` multiprocessors."""
    k, p = case.kind, case.p
    if k == "serial":
        return dict(blocks=_cdiv(p["n"], 64), tail=p["n"] % 64)
    if k == "scan":
        grid = min(_cdiv(p["n"] * 32, 128), sms * 16)
        return dict(grid_stride=p["n"] > 4 * grid, chunks=_cdiv(p["t"], 32), last_chunk=p["t"] % 32 or 32)
    if k == "backup":
        return dict(tail=p["n"] * p["d"] % 256)
    if k == "pc":
        h, w = p["hw"]
        c, cell = PLANE_C[p["plane"]], p["cell"]
        oh, ow = p["out"] or (h // cell, w // cell)
        smem = 2 * _pad16(h * w * c)
        return dict(smem_fits=smem <= SMEM, ctas=_ctas_per_sm(smem, 4), list_grid=sms * _ctas_per_sm(smem, 4),
                    cells=oh * ow, table=(oh * ow) % 4 == 0, chunks=_cdiv(p["t"], K_CHUNK), t_mod_ahead=p["t"] % K_AHEAD,
                    pow2_pool=cell & (cell - 1) == 0, margins=((h - oh * cell) // 2, (w - ow * cell) // 2))
    if k == "rows":
        return dict(grid_stride=p["n"] > sms * 64, unrolled=p["row16"] > 96)
    if k == "aux":
        return dict(grid_stride=p["m"] > sms * 8, smem_fits=_pad16(p["hw"][0] * p["hw"][1] * PLANE_C[p["plane"]]) <= SMEM)
    if k == "f32":
        h, w = p["hw"]
        c = PLANE_C[p["plane"]]
        vec = (h * w) % 4 == 0 and not p.get("off4")
        if vec:
            total = p["n"] * (h * w // 4)
            grid = min(_cdiv(total, 4 * 256), sms * 16)
            return dict(kernel="vec<%d>" % c, passes=_cdiv(total, 4 * 256 * grid), partial=total % (4 * 256 * grid) != 0)
        return dict(kernel="staged", grid_stride=p["n"] > sms * 8)
    if k == "leaves":
        u = LEAF_UNROLL[len(p["leaves"]) - 1]
        total = p["n"] * (84 * 84 // 4)
        grid = min(_cdiv(total, u * 256), sms * 16)
        return dict(unroll=u, passes=_cdiv(total, u * 256 * grid))
    if k == "rp":
        blocks = _cdiv(p["n"], RP_BLOCK)
        return dict(scan=blocks > RP_SCAN_BLOCKS, scan_passes=_cdiv(blocks, 1024) if blocks > RP_SCAN_BLOCKS else 0)
    if k == "replay":
        L = p["L"]
        return dict(chunks=_cdiv(p["count"], 32), window_spans_chunks=L > 32 or (L > 1 and p["count"] > 32),
                    cap_mod_32=p["cap"] % 32, whole_warps=p["n"] % 4 == 0)
    raise AssertionError(k)


def _serial_cases():
    out = []
    for n in (1, 63, 64, 65):
        for t in (1, 2, 128, 1000):
            out.append(Case("serial_n%d_t%d" % (n, t), "serial", dict(n=n, t=t), dict(tail=n % 64),
                            "vn_nstep_returns_kernel: 64-thread blocks, n %% 64 = %d (%s); t = %d" %
                            (n % 64, "full last block" if n % 64 == 0 else "partial last block", t)))
    return out


def _scan_cases():
    out = [Case("scan_n37_t33", "scan", dict(n=37, t=33), dict(grid_stride=False, chunks=2, last_chunk=1),
                "scan: a full chunk then a 1-step chunk, 37 warps (< 4 * grid)")]
    for t in (1, 31, 32, 33, 64, 65, 200):
        out.append(Case("scan_gs_t%d" % t, "scan", dict(n=9473, t=t),
                        dict(grid_stride=True, chunks=_cdiv(t, 32), last_chunk=t % 32 or 32),
                        "scan: n = 9,473 > 4 warps * 148 * 16 blocks = 9,472 -> grid-stride; t = %d: %d chunk(s), "
                        "last of %d steps" % (t, _cdiv(t, 32), t % 32 or 32)))
    return out


def _backup_cases():
    return [Case("backup_d%d" % d, "backup", dict(n=37, t=9, d=d), dict(tail=37 * d % 256),
                 "vn_backup_kernel: n * d = %d, not a multiple of 256 -> a partial last block" % (37 * d))
            for d in (1, 3, 400, 1849)]


def _pc(id_, world, plane, cell, out, B, t, claims, why, jump=0.3, layout="batch"):
    return Case(id_, "pc", dict(world=world, hw=WORLDS[world][0], plane=plane, cell=cell, out=out, B=B, t=t,
                                jump=jump, layout=layout), claims, why)


# worlds: key -> (frame_hw, planes, family, scenes)
WORLDS = {
    "w84": ((84, 84), ("rgb", "depth", "segmentation"), "gym", 1),
    "w18x22": ((18, 22), ("rgb", "depth", "segmentation"), "gym", 1),
    "w30x50": ((30, 50), ("rgb", "depth"), "gym", 1),
    "w174": ((174, 174), ("rgb", "depth"), "gym", 1),
    "w190": ((190, 190), ("rgb",), "gym", 1),
    "two_scenes": ((30, 50), ("rgb", "segmentation"), "gym", 2),
    "simple": ((18, 22), ("rgb", "depth"), "simple", 1),
}

PC_CASES = [
    _pc("pc_rgb_c4_20x20", "w84", "rgb", 4, (20, 20), 6, 17, dict(pow2_pool=True, chunks=2, t_mod_ahead=1),
        "84^2 RGB, cell 4 (divisor 16 = 2^4), t 17: a 16-step chunk and a 1-step chunk"),
    _pc("pc_rgb_c3_oddcrop", "w84", "rgb", 3, (26, 24), 5, 16, dict(pow2_pool=False, margins=(3, 6), chunks=1,
                                                                     t_mod_ahead=0, table=True),
        "cell 3 (divisor 9: a reciprocal multiply differs), 624 cells (table), top margin 3 (84 - 78 = 6, odd half), "
        "t = kChunk"),
    _pc("pc_depth_c5_oddcrop", "w84", "depth", 5, (15, 13), 4, 15, dict(pow2_pool=False, margins=(4, 9),
                                                                        t_mod_ahead=3, table=False),
        "1-channel plane, cell 5 (divisor 25), margins 4 and 9 (84 - 75, 84 - 65: odd differences), 195 cells "
        "(direct only), t 15 = 3 mod kAhead"),
    _pc("pc_seg_c8_none", "w84", "segmentation", 8, None, 4, 2, dict(cells=100, margins=(2, 2), t_mod_ahead=2),
        "segmentation, cell 8, output None -> 10 x 10 (100 cells), t 2 = 2 mod kAhead"),
    _pc("pc_rgb_c2_2x2", "w84", "rgb", 2, (2, 2), 3, 33, dict(cells=4, table=True, chunks=3, t_mod_ahead=1),
        "cell 2, 2 x 2 output: 4 cells, the smallest table row (one float4 per env and step); t 33: three chunks"),
    _pc("pc_rgb_c5_1x1", "w84", "rgb", 5, (1, 1), 3, 1, dict(cells=1, table=False, chunks=1),
        "1 x 1 output: 1 cell, not a multiple of 4 -> direct only (returns via discounted_backup); t 1"),
    _pc("pc_rgb_c4_t15", "w84", "rgb", 4, (20, 20), 7, 15, dict(table=True, chunks=1, t_mod_ahead=3),
        "table path at t 15 = 3 mod kAhead: the fused back-up's first 4-step group has one empty slot"),
    _pc("pc_depth_c4_t1", "w84", "depth", 4, (20, 20), 9, 1, dict(table=True, chunks=1, t_mod_ahead=1),
        "table path at t 1: one step, three empty kAhead slots, one direct-kernel chunk of 1 step"),
    _pc("pc_n1", "w84", "depth", 3, (28, 28), 1, 17, dict(cells=784, table=True),
        "n = 1 env, 1-channel, cell 3, 28 x 28 = 784 cells"),
    _pc("pc_time_major", "w84", "rgb", 4, (20, 20), 37, 16, dict(chunks=1),
        "states a .t() view of time-major [T+1, B] storage (the lookup kernel orders its threads env-fastest)",
        layout="time"),
    _pc("pc_many_misses", "w84", "rgb", 4, (20, 20), 64, 17, dict(list_grid=148 * 4, ctas=4),
        "every transition a random jump: ~1,000 misses > the list kernel's grid 148 * min(4, 225,280 // 43,360) = 592",
        jump=1.0),
    _pc("pc_18x22_c3", "w18x22", "rgb", 3, (4, 6), 5, 17, dict(margins=(3, 2), table=True),
        "non-square 18 x 22, cell 3, 4 x 6 (24 cells) with margins 3 and 2"),
    _pc("pc_18x22_seg_c2", "w18x22", "segmentation", 2, None, 5, 15, dict(cells=99, table=False),
        "18 x 22 segmentation, cell 2, None -> 9 x 11 = 99 cells (direct only)"),
    _pc("pc_30x50_c5", "w30x50", "rgb", 5, None, 5, 16, dict(cells=60, table=True, margins=(0, 0)),
        "non-square 30 x 50, cell 5, None -> 6 x 10"),
    _pc("pc_30x50_depth_c4", "w30x50", "depth", 4, (7, 12), 4, 33, dict(margins=(1, 1), table=True),
        "30 x 50 depth, cell 4, 7 x 12 with margins 1 and 1"),
    _pc("pc_174_c4", "w174", "rgb", 4, (42, 42), 3, 17, dict(ctas=1, cells=1764, margins=(3, 3)),
        "174^2 -> 42 x 42 (the reference's native frames), 2 * 90,832 B: 1 CTA per SM"),
    _pc("pc_190_limit", "w190", "rgb", 4, (46, 46), 2, 16, dict(smem_fits=True, ctas=1),
        "190^2 RGB: 2 * 108,304 = 216,608 B <= kMaxSmem 225,280 B, 1 CTA per SM"),
    _pc("pc_two_scenes", "two_scenes", "segmentation", 3, (10, 16), 8, 17, dict(table=True),
        "two scenes in one store (global state indices), cell 3"),
    _pc("pc_simple_graph", "simple", "rgb", 2, (8, 10), 8, 17, dict(table=True),
        "SIMPLE_GRAPH (unoriented: one state per cell, compass moves), cell 2"),
]


def _rows_cases():
    out = []
    for row16, n in ((1, 9473 * 2), (100, 9480), (300, 2000), (441, 9474)):
        out.append(Case("rows_u%d_n%d" % (row16, n), "rows", dict(row16=row16, n=n),
                        dict(grid_stride=n > 9472, unrolled=row16 > 96),
                        "vn_gather_rows: %d rows vs 148 * 64 = 9,472 warps; %d 16-byte units (%s)" %
                        (n, row16, "4-load loop" if row16 > 96 else "tail loop only")))
    return out


AUX_CASES = [
    Case("aux_depth_c5_2d", "aux", dict(plane="depth", cell=5, out=(16, 16), hw=(84, 84), m=1280, shape="2d"),
         dict(grid_stride=True), "c 1, cell 5, m = 1,280 > 148 * 8 = 1,184 frames; a [32, 40] .t() view"),
    Case("aux_seg_c3_1d", "aux", dict(plane="segmentation", cell=3, out=None, hw=(84, 84), m=1300, shape="1d"),
         dict(grid_stride=True), "c 3, cell 3 -> 28 x 28, m 1,300 > 1,184; 1-D states"),
    Case("aux_rgb_c4_3d", "aux", dict(plane="rgb", cell=4, out=(20, 20), hw=(84, 84), m=1300, shape="3d"),
         dict(grid_stride=True), "c 3, cell 4, 3-D [5, 20, 13] states"),
    Case("aux_depth_c2_small", "aux", dict(plane="depth", cell=2, out=(41, 41), hw=(84, 84), m=12, shape="2d"),
         dict(grid_stride=False), "c 1, cell 2, 41 x 41 (1,681 cells: table rows not whole float4s -> direct)"),
]

F32_CASES = [
    Case("f32_vec1_84", "f32", dict(plane="depth", hw=(84, 84), n=1400), dict(kernel="vec<1>", passes=2, partial=True),
         "vec<1>: 1,400 * 1,764 groups > one pass of 4 * 256 * 148 * 16 = 2,424,832 -> 2 passes, the last partial"),
    Case("f32_vec3_84", "f32", dict(plane="rgb", hw=(84, 84), n=1400), dict(kernel="vec<3>", passes=2, partial=True),
         "vec<3>: as f32_vec1_84 for RGB"),
    Case("f32_vec3_small", "f32", dict(plane="rgb", hw=(84, 84), n=3), dict(kernel="vec<3>", passes=1),
         "vec<3>: 3 frames, one partial pass"),
    Case("f32_staged_83", "f32", dict(plane="depth", hw=(83, 83), n=1190), dict(kernel="staged", grid_stride=True),
         "staged: 83 * 83 = 6,889 pixels (mod 4 = 1), 1,190 frames > 148 * 8 = 1,184 CTAs"),
    Case("f32_staged_18x21", "f32", dict(plane="rgb", hw=(18, 21), n=1300), dict(kernel="staged", grid_stride=True),
         "staged: 18 * 21 = 378 pixels (mod 4 = 2), RGB, 1,300 frames"),
    Case("f32_staged_off4", "f32", dict(plane="rgb", hw=(84, 84), n=40, off4=True), dict(kernel="staged"),
         "staged: a 4-byte-offset output (not 16-byte aligned) through the C ABI"),
]

LEAF_SETS = (
    (("rgb", 0),),
    (("depth", 1), ("rgb", 0)),
    (("segmentation", 1), ("depth", 0), ("rgb", 1)),
    (("rgb", 0), ("depth", 1), ("segmentation", 0), ("depth", 0)),
    (("depth", 1), ("rgb", 1), ("depth", 0), ("segmentation", 1), ("rgb", 0)),
    (("rgb", 1), ("depth", 0), ("segmentation", 0), ("depth", 1), ("rgb", 0), ("segmentation", 1)),
)
LEAF_CASES = [Case("leaves%d" % len(ls), "leaves", dict(leaves=ls, n=360),
                   dict(unroll=LEAF_UNROLL[len(ls) - 1], passes=_cdiv(360 * 1764, LEAF_UNROLL[len(ls) - 1] * 256 * 2368)),
                   "vn_gather_leaves_f32_kernel<%d, %d>: 360 frames of 1,764 groups; channels %s, sources %s"
                   % (len(ls), LEAF_UNROLL[len(ls) - 1], [PLANE_C[p] for p, _ in ls], [s for _, s in ls]))
              for ls in LEAF_SETS]

RP_CASES = [Case("rp_n%d" % n, "rp", dict(n=n), dict(scan=n > 256 * 1024, scan_passes=_cdiv(_cdiv(n, 1024), 1024)
                                                      if n > 256 * 1024 else 0),
                 "RP: %d blocks of 1,024 (%s)" % (_cdiv(n, 1024), why))
            for n, why in ((1, "one partial block"), (1023, "one partial block"), (1024, "one whole block"),
                           (1025, "a whole and a 1-element block"), (262144, "256 blocks: the last unscanned size"),
                           (262145, "257 blocks: the first scanned size"), (1 << 20, "1,024 blocks: one scan pass"),
                           ((1 << 20) + 1, "1,025 blocks: two scan passes"), (1 << 24, "16,384 blocks: 16 scan passes"))]
RP_CASES.append(Case("rp_time_major", "rp", dict(n=100 * 10500, t=100), dict(scan=True, scan_passes=2),
                     "RP: a [10,500, 100] .t() view of time-major storage (t = 100 does not divide 1,024), 1,026 "
                     "blocks: two scan passes"))


def _replay(id_, L, cap, count, n=37, p_done=0.06, claims=None, why="", base=0, seed=7, mode=0):
    return Case(id_, "replay", dict(L=L, cap=cap, count=count, n=n, p_done=p_done, base=base, seed=seed, mode=mode),
                claims or {}, why)


REPLAY_CASES = [
    _replay("replay_L1", 1, 96, 96, claims=dict(chunks=3), why="L 1: every transition is a window"),
    _replay("replay_L31", 31, 96, 90, claims=dict(chunks=3), why="L 31: windows cross 32-slot chunks"),
    _replay("replay_L32", 32, 96, 96, claims=dict(window_spans_chunks=True), why="L 32 = one chunk"),
    _replay("replay_L33", 33, 100, 100, claims=dict(cap_mod_32=4, window_spans_chunks=True),
            why="L 33 > a chunk; cap 100 not a multiple of 32"),
    _replay("replay_L40_wrap", 40, 75, 75, claims=dict(cap_mod_32=11, chunks=3),
            why="L 40, cap 75 (mod 32 = 11), full ring, head mid-ring: the column wraps"),
    _replay("replay_L_cap", 50, 50, 50, p_done=0.01, claims=dict(chunks=2),
            why="L = cap: at most one window (rare episode ends, so most envs have it)"),
    _replay("replay_count_lt_L", 33, 64, 20, claims=dict(chunks=1), why="count 20 < L 33: no window"),
    _replay("replay_all_done", 4, 70, 70, p_done=1.0, why="every transition ends an episode: no window of 4"),
    _replay("replay_no_done", 33, 70, 70, p_done=0.0, why="no episode end: every in-ring window valid"),
    _replay("replay_base_seed", 33, 100, 90, n=37, base=1000, seed=0x9E3779B97F4A7C15,
            claims=dict(whole_warps=False), why="n 37 (mod 4 = 1), env_id_base 1,000, seed with its high 32 bits set"),
    _replay("replay_rp_mode", 4, 100, 100, p_done=0.1, mode=1, claims=dict(chunks=4),
            why="RP mode: 3 history steps + the classified one, zero / non-zero classes"),
]

CASES = (_serial_cases() + _scan_cases() + _backup_cases() + PC_CASES + _rows_cases() + AUX_CASES + F32_CASES +
         LEAF_CASES + RP_CASES + REPLAY_CASES)


def _of(kind):
    return [c for c in CASES if c.kind == kind]


# ---------------------------------------------------------------- CPU check of the case table
def _check_claims(case, sms):
    plan = _plan(case, sms)
    assert {k: plan[k] for k in case.claims} == case.claims, (case.id, plan)


def test_case_table_branches():
    """Every case lands on the launch branch its name and derivation claim, on a B200 (148 SMs)."""
    assert len({c.id for c in CASES}) == len(CASES)
    for case in CASES:
        _check_claims(case, B200_SMS)
    # the edges the table is built around
    assert _plan(_of("scan")[1], B200_SMS)["grid_stride"] and not _plan(_of("scan")[0], B200_SMS)["grid_stride"]
    pcs = {c.id: _plan(c, B200_SMS) for c in PC_CASES}
    assert pcs["pc_190_limit"]["smem_fits"] and pcs["pc_190_limit"]["ctas"] == 1
    assert {c.p["cell"] for c in PC_CASES} >= {2, 3, 4, 5, 8}
    assert {c.p["plane"] for c in PC_CASES} == set(PLANE_C)
    fused = [c for c in PC_CASES if pcs[c.id]["table"]]      # the cases that run vn_pc_returns_kernel
    assert {c.p["t"] % K_AHEAD for c in fused} == {0, 1, 2, 3}
    assert {c.p["t"] for c in fused} >= {1, 15, 16, 17, 33}
    rp = {c.p["n"]: _plan(c, B200_SMS) for c in RP_CASES}
    assert not rp[262144]["scan"] and rp[262145]["scan"] and rp[1 << 20]["scan_passes"] == 1
    assert rp[(1 << 20) + 1]["scan_passes"] == 2
    assert sorted(len(c.p["leaves"]) for c in LEAF_CASES) == [1, 2, 3, 4, 5, 6]
    assert {c.p["L"] for c in REPLAY_CASES} >= {1, 31, 32, 33, 40}


# ---------------------------------------------------------------- GPU side
def _torch():
    import torch
    return torch


def _sms():
    torch = _torch()
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _ready(case):
    """The case's branch, recomputed for this device: a GPU with another SM count must not pass without reaching it."""
    _check_claims(case, _sms())


def _rng(case_id):
    return np.random.RandomState(zlib.crc32(case_id.encode()))


@lru_cache(maxsize=None)
def _world(key):
    hw, planes, fam, nscenes = WORLDS[key]
    T = vn.tables
    oriented = fam == "gym"
    scenes = [vn.scenes.make_maze_scene((8, 9), 0.25, 3 + i, n_goals=1, oriented=oriented, frame_hw=hw, planes=planes,
                                        scene_id=i) for i in range(nscenes)]
    return vn.DeviceWorld(T.compile_world(scenes, T.GYM_GRAPH if oriented else T.SIMPLE_GRAPH))


@lru_cache(maxsize=None)
def _byte_world(hw, planes):
    """A world whose frames are explicit random bytes, each frame holding all 256 byte values."""
    scene = vn.scenes.make_maze_scene((6, 7), 0.2, 11, frame_hw=hw, planes=planes)
    rng = np.random.RandomState(hw[0] * 1000 + hw[1])
    explicit = {}
    for p in planes:
        a = rng.randint(0, 256, size=(scene.n_states, hw[0] * hw[1] * PLANE_C[p])).astype(np.uint8)
        a[:, :256] = np.arange(256, dtype=np.uint8)[None]
        a[:, :256] = a[:, rng.permutation(256)]
        explicit[p] = a.reshape(scene.n_states, hw[0], hw[1], PLANE_C[p])
    scene.explicit = explicit
    return vn.DeviceWorld(vn.tables.compile_world([scene], vn.tables.GYM_GRAPH))


def _walk(world, B, T1, jump, rng):
    """[B, T1] state sequences: moves along the adjacency (a collision keeps the state) with a random jump (a reset,
    which the transition table cannot serve) at probability `jump`."""
    S, adj = world.n_states, world.adj
    st = np.empty((B, T1), np.int32)
    st[:, 0] = rng.randint(0, S, B)
    for k in range(1, T1):
        nxt = adj[st[:, k - 1], rng.randint(0, 4, B)]
        nxt = np.where(nxt >= 0, nxt, st[:, k - 1])
        st[:, k] = np.where(rng.rand(B) < jump, rng.randint(0, S, B), nxt)
    return st


def _misses(world, st):
    """[B, T] bool: transition st[:, k] -> st[:, k + 1] is neither a repeat nor an adjacency entry."""
    a, b = st[:, :-1], st[:, 1:]
    return (a != b) & ~(world.adj[a] == b[..., None]).any(-1)


def _bits(x):
    torch = _torch()
    if torch.is_tensor(x):
        x = x.detach().cpu().numpy()
    x = np.ascontiguousarray(x)
    return x.view(np.uint32) if x.dtype == np.float32 else x


def _same(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    if np.array_equal(g, w):
        return
    bad = np.argwhere(g != w)
    raise AssertionError("%s: %d of %d elements differ, first at %s" % (what, len(bad), g.size, bad[0].tolist()))


def _states_tensor(st, layout):
    torch = _torch()
    if layout == "time":
        return torch.from_numpy(np.ascontiguousarray(st.T)).cuda().t()
    return torch.from_numpy(st).cuda()


# ---------------------------------------------------------------- n-step returns, back-up
@pytest.mark.gpu
@pytest.mark.parametrize("time_major", [False, True], ids=["batch", "time"])
@pytest.mark.parametrize("case", _of("serial"), ids=lambda c: c.id)
def test_serial_returns_bit_equal(case, time_major):
    torch = _torch()
    _ready(case)
    n, t = case.p["n"], case.p["t"]
    rng = _rng(case.id)
    r = rng.randn(n, t).astype(np.float32)
    d = rng.rand(n, t) < 0.1
    v = rng.randn(n).astype(np.float32)
    want = orl.nstep_returns(r, d, v, 0.99)
    rt, dt, vt = torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda(), torch.from_numpy(v).cuda()
    if time_major:
        got = vn.rollout.nstep_returns(rt.t().contiguous(), dt.t().contiguous(), vt, 0.99, time_major=True).t()
    else:
        got = vn.rollout.nstep_returns(rt, dt, vt, 0.99)
    _same(got, want, case.id)


def _returns64(r, d, v, gamma):
    """float64 R_t = r_t + gamma (1 - done_t) R_{t+1}, R_T = (1 - done_{T-1}) V, and the same recurrence on |r|, |V|."""
    n, t = r.shape
    nd = 1.0 - d.astype(np.float64)
    out, mag = np.zeros((n, t)), np.zeros((n, t))
    R = nd[:, -1] * v.astype(np.float64)
    M = np.abs(R)
    for k in reversed(range(t)):
        R = r[:, k] + gamma * nd[:, k] * R
        M = np.abs(r[:, k]) + gamma * nd[:, k] * M
        out[:, k], mag[:, k] = R, M
    return out, mag


def _scan_bound(t, mag):
    """Error bound of the warp scan: per 32-step chunk, 5 shuffle levels each round the map's slope (a * a2) and
    offset (one fma), and one fma applies the chunk's map to the carry; the carry chain crosses ceil(t / 32) chunks.
    So every term of R_t goes through at most (2 * 5 + 1) * ceil(t / 32) + 1 roundings (the + 1: the bootstrap
    product), each a relative error of at most 2^-24 of a partial sum bounded by the |r| recurrence."""
    m = (2 * 5 + 1) * _cdiv(t, 32) + 1
    u = 2.0 ** -24
    return m * u / (1 - m * u) * mag


@pytest.mark.gpu
@pytest.mark.parametrize("time_major", [False, True], ids=["batch", "time"])
@pytest.mark.parametrize("case", _of("scan"), ids=lambda c: c.id)
def test_scan_returns_within_bound(case, time_major):
    """method="scan" against a float64 recurrence, within the scan's operation-count bound; the bound rejects a dropped
    done flag, gamma applied once too often at a chunk boundary, and rewards shifted by one step."""
    torch = _torch()
    _ready(case)
    n, t, gamma = case.p["n"], case.p["t"], 0.99
    rng = _rng(case.id)
    r = rng.randn(n, t).astype(np.float32)
    d = rng.rand(n, t) < 0.05
    v = rng.randn(n).astype(np.float32)
    rt, dt = torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda()
    if time_major:
        rt, dt = rt.t().contiguous(), dt.t().contiguous()
    got = vn.rollout.nstep_returns(rt, dt, torch.from_numpy(v).cuda(), gamma, time_major=time_major, method="scan")
    got = (got.t() if time_major else got).cpu().numpy().astype(np.float64)
    ref, mag = _returns64(r.astype(np.float64), d, v, np.float64(np.float32(gamma)))
    bound = _scan_bound(t, mag)
    err = np.abs(got - ref)
    ratio = float((err / np.maximum(bound, 1e-300)).max())
    print("%s %s: worst |scan - float64| / bound = %.4f" % (case.id, "time" if time_major else "batch", ratio))
    assert (err <= bound).all(), ratio
    if time_major or t < 33:
        return
    g = np.float64(np.float32(gamma))
    wrongs = {}
    cand = np.argwhere(d[:, :-1])                                      # done flags before the last step
    e, k = cand[np.argmax(np.abs(ref[cand[:, 0], cand[:, 1] + 1]))]   # the one whose drop changes R most
    d2 = d.copy()
    d2[e, k] = False
    wrongs["dropped done"] = _returns64(r.astype(np.float64), d2, v, g)[0]
    hi = t - 32                                                        # first step of the last full chunk
    w = ref.copy()
    w[:, hi - 1] = r[:, hi - 1] + g * g * (1 - d[:, hi - 1]) * ref[:, hi]   # the carry scaled by gamma twice
    wrongs["extra gamma at a chunk boundary"] = w
    wrongs["rewards shifted one step"] = _returns64(np.roll(r, 1, 1).astype(np.float64), d, v, g)[0]
    for what, wrong in wrongs.items():
        assert not (np.abs(wrong - ref) <= bound).all(), what


@pytest.mark.gpu
@pytest.mark.parametrize("case", _of("backup"), ids=lambda c: c.id)
def test_discounted_backup_bit_equal(case):
    torch = _torch()
    _ready(case)
    n, t, dd = case.p["n"], case.p["t"], case.p["d"]
    rng = _rng(case.id)
    r = rng.rand(n, t, dd).astype(np.float32)
    d = rng.rand(n, t) < 0.2
    b = rng.randn(n, dd).astype(np.float32)
    want = orl.discounted_backup(r, d, b, 0.9)
    dones = torch.from_numpy(np.ascontiguousarray(d.T)).cuda().t()      # [n, t] view of time-major storage
    got = vn.rollout.discounted_backup(torch.from_numpy(r).cuda(), dones, torch.from_numpy(b).cuda(), 0.9)
    _same(got, want, case.id)


# ---------------------------------------------------------------- pixel control
def _pc_inputs(case):
    p = case.p
    dw = _world(p["world"])
    rng = _rng(case.id)
    st = _walk(dw.world, p["B"], p["t"] + 1, p["jump"], rng)
    return dw, st, rng


def _pc_oracle(dw, st, plane, cell, out):
    torch = _torch()
    fr = dw.plane_view(plane)[torch.from_numpy(st.reshape(-1)).cuda().long()].cpu().numpy()
    fr = fr.reshape(st.shape + fr.shape[1:])
    return orl.pixel_control_reward(orl.u8_to_policy_input(fr), cell, out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PC_CASES, ids=lambda c: c.id)
def test_pixel_control_paths_bit_equal(case):
    """direct == oracle (on up to 8 sampled envs), table (rows + list kernel) == direct, and the fused returns with
    and without the rewards == the oracle back-up of the direct rewards, all bit for bit."""
    torch = _torch()
    _ready(case)
    p = case.p
    dw, st, rng = _pc_inputs(case)
    plane, cell, out = p["plane"], p["cell"], p["out"]
    states = _states_tensor(st, p["layout"])
    direct = vn.rollout.pixel_control_reward(dw, states, cell, out, plane, method="direct")
    B, t = st.shape[0], st.shape[1] - 1
    sample = np.sort(rng.choice(B, size=min(B, 8), replace=False))
    _same(direct[torch.from_numpy(sample).cuda()], _pc_oracle(dw, st[sample], plane, cell, out), "direct vs oracle")
    miss = _misses(dw.world, st)
    plan = _plan(case, _sms())
    if case.id == "pc_many_misses":
        assert miss.sum() > plan["list_grid"]
    table = vn.rollout.pixel_control_reward(dw, states, cell, out, plane, method="table")
    _same(table, direct, "table vs direct")
    assert bool((direct[torch.from_numpy(st[:, 1:] == st[:, :-1]).cuda()] == 0).all())
    cells = plan["cells"]
    d = rng.rand(B, t) < 0.2
    boot = rng.rand(B, cells).astype(np.float32)
    dones = torch.from_numpy(np.ascontiguousarray(d.T)).cuda().t() if p["layout"] == "time" else torch.from_numpy(d).cuda()
    ret, rew = vn.rollout.pixel_control_returns(dw, states, dones, torch.from_numpy(boot).cuda(), 0.9, cell, out, plane,
                                                with_reward=True)
    _same(rew, direct.view(B, t, cells), "fused rewards vs direct")
    want = orl.discounted_backup(direct.view(B, t, cells).cpu().numpy(), d, boot, 0.9)
    _same(ret, want, "fused returns vs oracle back-up")
    _same(vn.rollout.pixel_control_returns(dw, states, dones, torch.from_numpy(boot).cuda(), 0.9, cell, out, plane),
          want, "fused returns without rewards")


@pytest.mark.gpu
def test_max_miss_overflow_gives_nan_and_leaves_the_rest_bit_identical():
    """max_miss below the number of table misses: exactly misses - max_miss reward rows are NaN, all at miss positions
    (which ones is up to the device's atomic); a return is NaN exactly where an overflowed transition lies at or after
    it in its env; every other element equals the unbounded call bit for bit."""
    torch = _torch()
    dw = _world("w84")
    rng = np.random.RandomState(5)
    B, t, cells = 24, 17, 400
    st = _walk(dw.world, B, t + 1, 0.15, rng)
    miss = _misses(dw.world, st)
    n_miss = int(miss.sum())
    states = torch.from_numpy(st).cuda()
    dones = torch.from_numpy(rng.rand(B, t) < 0.2).cuda()
    boot = torch.rand(B, cells, device="cuda")
    ret0, rew0 = vn.rollout.pixel_control_returns(dw, states, dones, boot, 0.9, 4, (20, 20), with_reward=True)
    for k in (1, n_miss // 2, n_miss - 1):
        ret, rew = vn.rollout.pixel_control_returns(dw, states, dones, boot, 0.9, 4, (20, 20), with_reward=True,
                                                    max_miss=k)
        nan_rows = torch.isnan(rew).all(-1).cpu().numpy()
        assert not (torch.isnan(rew).any(-1).cpu().numpy() & ~nan_rows).any()
        assert nan_rows.sum() == n_miss - k and not (nan_rows & ~miss).any()
        tail = np.flip(np.logical_or.accumulate(np.flip(nan_rows, 1), 1), 1)    # an overflow at or after (env, step)
        ret_nan = torch.isnan(ret).cpu().numpy()
        assert (ret_nan == tail[..., None]).all()
        keep = torch.from_numpy(~nan_rows).cuda()
        _same(rew[keep], rew0[keep], "rewards outside the overflow")
        keep = torch.from_numpy(~tail).cuda()
        _same(ret[keep], ret0[keep], "returns outside the overflow")
    assert n_miss > 3


# ---------------------------------------------------------------- row gather
@pytest.mark.gpu
@pytest.mark.parametrize("case", _of("rows"), ids=lambda c: c.id)
def test_gather_rows_bit_equal(case):
    """vn_gather_rows: idx >= 0 copies the row, -1 writes zeros, <= -2 leaves the row untouched (sentinel bytes)."""
    torch = _torch()
    _ready(case)
    row16, n = case.p["row16"], case.p["n"]
    gen = torch.Generator(device="cuda").manual_seed(zlib.crc32(case.id.encode()))
    R, T = 97, 8 if n % 8 == 0 else (2 if n % 2 == 0 else 1)
    table = torch.randint(-2 ** 31, 2 ** 31 - 1, (R, row16 * 4), dtype=torch.int32, device="cuda", generator=gen)
    idx = torch.randint(-4, R, (T, n // T), dtype=torch.int32, device="cuda", generator=gen)   # time-major storage
    view = idx.t()                                                                           # [n / T, T] view
    out = torch.full((n, row16 * 4), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    lib = vn.lib.load()
    vn.lib.check(lib.vn_gather_rows(table.data_ptr(), row16 * 16, view.data_ptr(), n, T, view.stride(0), view.stride(1),
                                    out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    flat = view.reshape(-1).long()
    want = torch.where((flat >= 0)[:, None], table[flat.clamp_min(0)], torch.zeros_like(table[:1]))
    want = torch.where((flat <= -2)[:, None], torch.full_like(want, 0x5A5A5A5A), want)
    assert bool((flat == -1).any()) and bool((flat <= -2).any())
    _same(out, want, case.id)


# ---------------------------------------------------------------- aux targets
@pytest.mark.gpu
@pytest.mark.parametrize("case", AUX_CASES, ids=lambda c: c.id)
def test_aux_targets_bit_equal(case):
    """direct == oracle on 64 sampled frames, table == direct in full."""
    torch = _torch()
    _ready(case)
    p = case.p
    dw = _world("w84")
    rng = _rng(case.id)
    m, S = p["m"], dw.world.n_states
    flat = rng.randint(0, S, m).astype(np.int32)
    if p["shape"] == "1d":
        states = torch.from_numpy(flat).cuda()
    elif p["shape"] == "3d":
        states = torch.from_numpy(flat.reshape(5, 20, 13)).cuda()
    else:
        b = 32 if m % 32 == 0 else m
        states = torch.from_numpy(flat.reshape(m // b, b)).cuda().t()      # [b, m / b] .t() view
    direct = vn.rollout.auxiliary_target(dw, states, p["plane"], p["cell"], p["out"], method="direct")
    table = vn.rollout.auxiliary_target(dw, states, p["plane"], p["cell"], p["out"], method="table")
    _same(table, direct, "table vs direct")
    flat_view = states.reshape(-1).cpu().numpy()
    sample = np.sort(rng.choice(m, size=min(m, 64), replace=False))
    fr = dw.plane_view(p["plane"])[torch.from_numpy(flat_view[sample]).cuda().long()].cpu().numpy()
    want = orl.aux_target(orl.u8_to_policy_input(fr[None]), p["cell"], p["out"])[0]
    _same(direct.reshape((m,) + direct.shape[states.dim():])[torch.from_numpy(sample).cuda()], want, "direct vs oracle")


@pytest.mark.gpu
def test_aux_target_on_a_depth_only_world_builds_no_pixel_control_table():
    torch = _torch()
    scene = vn.scenes.make_maze_scene((6, 6), 0.2, 2, planes=("depth",))
    dw = vn.DeviceWorld(vn.tables.compile_world([scene], vn.tables.GYM_GRAPH))
    states = torch.randint(0, dw.world.n_states, (4, 9), dtype=torch.int32, device="cuda")
    got = vn.rollout.auxiliary_target(dw, states, "depth", 4, (20, 20))
    assert not dw.__dict__.get("_target_tables")
    _same(got, vn.rollout.auxiliary_target(dw, states, "depth", 4, (20, 20), method="direct"), "table vs direct")


# ---------------------------------------------------------------- float gathers
LUT = (np.arange(256).astype(np.float32) / np.float32(255)).astype(np.float32)


SENTINEL = 0x7FC5A5A5     # bits of a quiet NaN no kernel writes


def _sentinel(shape):
    torch = _torch()
    return torch.full(shape, SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


def _chw_expected(dw, plane, recs, untouched):
    """float32 [n, C, H, W]: LUT[byte] of record recs[i], or the sentinel where recs[i] < 0 (untouched) / zeros."""
    torch = _torch()
    lut = torch.from_numpy(LUT).cuda()
    recs = torch.as_tensor(recs, device="cuda").long()
    fr = dw.plane_view(plane)[recs.clamp_min(0)]
    want = lut[fr.long()].permute(0, 3, 1, 2)
    other = _sentinel(want.shape) if untouched else torch.zeros_like(want)
    return torch.where((recs >= 0)[:, None, None, None], want, other)


@pytest.mark.gpu
@pytest.mark.parametrize("case", F32_CASES, ids=lambda c: c.id)
def test_float_gathers_bit_equal(case):
    """policy_input / vn_gather_plane_f32_chw[_rows] == u8.astype(f32) / f32(255) bit for bit on frames holding all 256
    byte values; the rows variant leaves rows with a negative index untouched; nothing is written outside."""
    torch = _torch()
    _ready(case)
    p = case.p
    plane, (h, w), n = p["plane"], p["hw"], p["n"]
    dw = _byte_world(tuple(p["hw"]), ("rgb", "depth"))
    c = PLANE_C[plane]
    rng = _rng(case.id)
    recs = rng.randint(0, dw.world.n_states, n).astype(np.int32)
    if not p.get("off4"):
        got = vn.rollout.policy_input(dw, torch.from_numpy(recs), plane)
        _same(got, _chw_expected(dw, plane, recs, False), "policy_input")
    lib, stream = vn.lib.load(), torch.cuda.current_stream().cuda_stream
    shift = 1 if p.get("off4") else 4          # 4 bytes or 16 bytes into the buffer
    size = n * c * h * w
    buf = _sentinel((shift + size + 4,))
    idx = torch.from_numpy(np.stack([recs, np.where(rng.rand(n) < 0.25, -1, recs)], 1).astype(np.int32)).cuda()
    idx[::7, 1] = -1
    vn.lib.check(lib.vn_gather_plane_f32_chw_rows(C.byref(dw.store), dw.plane_index(plane), idx[:, 1:].data_ptr(), 2, n,
                                                  h, w, c, buf[shift:].data_ptr(), stream))
    _same(buf[shift:shift + size].view(n, c, h, w), _chw_expected(dw, plane, idx[:, 1], True), "rows variant")
    _same(buf[:shift], _sentinel((shift,)), "before the output")
    _same(buf[shift + size:], _sentinel((4,)), "after the output")


@pytest.mark.gpu
@pytest.mark.parametrize("case", LEAF_CASES, ids=lambda c: c.id)
def test_float_leaves_bit_equal(case):
    """vn_gather_leaves_f32_chw: every leaf == LUT[byte] of its record (descriptor x or y), untouched where it is -1."""
    torch = _torch()
    _ready(case)
    n, leaves = case.p["n"], case.p["leaves"]
    dw = _byte_world((84, 84), ("rgb", "depth", "segmentation"))
    rng = _rng(case.id)
    S = dw.world.n_states
    desc = rng.randint(0, S, (n, 2)).astype(np.int32)
    desc[rng.rand(n) < 0.2, 0] = -1
    desc[rng.rand(n) < 0.2, 1] = -1
    desc_t = torch.from_numpy(desc).cuda()
    outs = [_sentinel((n, PLANE_C[pl], 84, 84)) for pl, _ in leaves]
    arr = (vn.lib.FloatLeaf * len(leaves))()
    for i, ((pl, src), o) in enumerate(zip(leaves, outs)):
        arr[i].plane, arr[i].source, arr[i].channels, arr[i].out = dw.plane_index(pl), src, PLANE_C[pl], o.data_ptr()
    vn.lib.check(vn.lib.load().vn_gather_leaves_f32_chw(C.byref(dw.store), arr, len(leaves), desc_t.data_ptr(), n, 84, 84,
                                                        torch.cuda.current_stream().cuda_stream))
    for (pl, src), o in zip(leaves, outs):
        _same(o, _chw_expected(dw, pl, desc[:, src], True), "%s leaf from source %d" % (pl, src))


# ---------------------------------------------------------------- reward-prediction labels
def _rp_rewards(case):
    rng = _rng(case.id)
    n = case.p["n"]
    r = np.where(rng.rand(n) < 0.03, rng.choice([-1.0, 1.0, 0.5], size=n), 0.0).astype(np.float32)
    return r


def _check_rp(torch, r_dev, r_host):
    labels, zero, nonzero = vn.rollout.reward_prediction_labels(r_dev)
    z, nz = orl.rp_index_lists(r_host)
    _same(labels, orl.rp_labels(r_host), "labels")
    _same(zero, z, "zero list")
    _same(nonzero, nz, "non-zero list")
    l2, z2, nz2, counts = vn.rollout.reward_prediction_labels(r_dev, sync=False)
    _same(counts, np.array([len(z), len(nz)], np.int32), "counts")
    _same(l2, labels, "labels (sync=False)")
    _same(z2[:len(z)], z, "zero list (sync=False)")
    _same(nz2[:len(nz)], nz, "non-zero list (sync=False)")


@pytest.mark.gpu
@pytest.mark.parametrize("case", RP_CASES, ids=lambda c: c.id)
def test_rp_labels_and_lists_equal(case):
    torch = _torch()
    _ready(case)
    r = _rp_rewards(case)
    if "t" in case.p:
        t = case.p["t"]
        r2 = r.reshape(-1, t)
        dev = torch.from_numpy(np.ascontiguousarray(r2.T)).cuda().t()        # [B, t] view of time-major storage
        _check_rp(torch, dev, r2)
    else:
        _check_rp(torch, torch.from_numpy(r).cuda(), r)


@pytest.mark.gpu
@pytest.mark.parametrize("fill", ["zero", "nonzero", "special"])
def test_rp_labels_of_uniform_and_special_rewards(fill):
    """All-zero and all-non-zero rewards (one list empty), and -0.0 (zero class), denormals (non-zero, class 1 / 2),
    +-inf and NaN (non-zero list, label 0), across the scanned path."""
    torch = _torch()
    n = 262145
    rng = np.random.RandomState(17)
    if fill == "zero":
        r = np.zeros(n, np.float32)
    elif fill == "nonzero":
        r = rng.choice([-2.0, 0.25, 3.0], size=n).astype(np.float32)
    else:
        tiny = np.float32(1e-45)
        vals = np.array([0.0, -0.0, tiny, -tiny, np.float32(1e-40), np.inf, -np.inf, np.nan, 1.0], np.float32)
        r = vals[rng.randint(0, len(vals), n)]
    _check_rp(torch, torch.from_numpy(r).cuda(), r)


# ---------------------------------------------------------------- replay sampler
@pytest.mark.gpu
@pytest.mark.parametrize("case", REPLAY_CASES, ids=lambda c: c.id)
def test_replay_draws_equal_the_oracle(case):
    torch = _torch()
    _ready(case)
    p = case.p
    dw = _world("w84")
    rng = _rng(case.id)
    n, cap, count = p["n"], p["cap"], p["count"]
    ring = vn.rollout.ReplayRing(dw, n, capacity=cap, seed=p["seed"], env_id_base=p["base"])
    host = dict(before=rng.randint(0, 10 ** 6, (cap, n)), after=rng.randint(0, 10 ** 6, (cap, n)),
                goal=rng.randint(0, 10 ** 6, (cap, n)), goal_before=rng.randint(0, 10 ** 6, (cap, n)),
                action=rng.randint(0, 4, (cap, n)),
                reward=np.where(rng.rand(cap, n) < 0.3, rng.choice([-1.0, 1.0], (cap, n)), 0.0),
                done=rng.rand(cap, n) < p["p_done"])
    for k, v in host.items():
        getattr(ring, k).copy_(torch.from_numpy(v.astype(getattr(ring, k).cpu().numpy().dtype)))
    host = {k: getattr(ring, k).cpu().numpy() for k in host}
    ring.head, ring.count = (count + 13) % cap, count
    L = 4 if p["mode"] == 1 else p["L"]
    drawn = 0
    for _ in range(3):
        call = ring.calls
        smp = ring.sample_rp_sequence() if p["mode"] == 1 else ring.sample_sequence(L)
        got = {k: v.cpu().numpy() for k, v in smp.items()}
        oldest = (ring.head - count + cap) % cap
        for e in range(n):
            col = {k: v[:, e] for k, v in host.items()}
            want = orl.replay_sample(col["before"], col["after"], col["reward"], col["done"], ring.head, count, L,
                                     p["mode"], p["seed"], p["base"] + e, call, col["goal_before"], col["goal"])
            assert got["start"][e] == want[0], (e, got["start"][e], want[0])
            if want[0] < 0:
                continue
            drawn += 1
            slots = [(oldest + want[0] + k) % cap for k in range(L)]
            assert got["states"][e].tolist() == want[1] and got["goals"][e].tolist() == want[3], e
            assert got["actions"][e].tolist() == col["action"][slots].tolist()
            _same(got["rewards"][e], col["reward"][slots], "rewards")
            assert got["dones"][e].tolist() == col["done"][slots].tolist()
            if p["mode"] == 1:
                assert got["label"][e] == want[2]
    if case.id in ("replay_count_lt_L", "replay_all_done"):
        assert drawn == 0
    else:
        assert drawn > 0


# ---------------------------------------------------------------- empty batches
@pytest.mark.gpu
def test_empty_batches_return_empty_results_without_launching():
    """B = 0 with freshly allocated (null-pointer) tensors: every builder returns the documented empty shapes and
    launches no library kernel; so does RolloutBuffer(dw, 0, T).targets()."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    dw = _world("w84")
    R, T = vn.rollout, 5
    i32 = dict(dtype=torch.int32, device="cuda")
    f32 = dict(dtype=torch.float32, device="cuda")
    buf = R.RolloutBuffer(dw, 0, T)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = {
            "serial": R.nstep_returns(torch.empty((0, T), **f32), torch.empty((0, T), dtype=torch.uint8, device="cuda"),
                                      torch.empty(0, **f32), 0.99),
            "scan": R.nstep_returns(torch.empty((T, 0), **f32), torch.empty((T, 0), dtype=torch.bool, device="cuda"),
                                    torch.empty(0, **f32), 0.99, time_major=True, method="scan"),
            "backup": R.discounted_backup(torch.empty((0, T, 20, 20), **f32),
                                          torch.empty((0, T), dtype=torch.uint8, device="cuda"),
                                          torch.empty((0, 20, 20), **f32), 0.9),
            "pc_direct": R.pixel_control_reward(dw, torch.empty((0, T + 1), **i32), 4, (20, 20), method="direct"),
            "pc_table": R.pixel_control_reward(dw, torch.empty((0, T + 1), **i32), 4, (20, 20), method="table"),
            "pc_returns": R.pixel_control_returns(dw, torch.empty((0, T + 1), **i32),
                                                  torch.empty((0, T), dtype=torch.uint8, device="cuda"),
                                                  torch.empty((0, 400), **f32), 0.9, 4, (20, 20), with_reward=True),
            "aux_direct": R.auxiliary_target(dw, torch.empty((0, T), **i32), "depth", 4, (20, 20), method="direct"),
            "aux_table": R.auxiliary_target(dw, torch.empty((0, T), **i32), "segmentation", 4, (20, 20)),
            "policy_input": R.policy_input(dw, torch.empty(0, **i32)),
            "rp": R.reward_prediction_labels(torch.empty((0, T), **f32)),
            "rp_async": R.reward_prediction_labels(torch.empty((0, T), **f32), sync=False),
            "targets": buf.targets(torch.empty(0, **f32), 0.99, torch.empty((0, 400), **f32), 0.9, 4, (20, 20)),
            "targets_overlap": buf.targets(torch.empty(0, **f32), 0.99, torch.empty((0, 400), **f32), 0.9, 4, (20, 20),
                                           overlap=True),
        }
        torch.cuda.synchronize()
    launched = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert not any("vn_" in name for name in launched), launched
    shapes = {"serial": (0, T), "scan": (T, 0), "backup": (0, T, 20, 20), "pc_direct": (0, T, 1, 20, 20),
              "pc_table": (0, T, 1, 20, 20), "aux_direct": (0, T, 1, 20, 20), "aux_table": (0, T, 3, 20, 20),
              "policy_input": (0, 3, 84, 84)}
    for k, s in shapes.items():
        assert tuple(got[k].shape) == s, k
    assert [tuple(x.shape) for x in got["pc_returns"]] == [(0, T, 400)] * 2
    assert [tuple(x.shape) for x in got["rp"]] == [(0, T), (0,), (0,)]
    assert len(got["rp_async"]) == 4 and got["rp_async"][3].tolist() == [0, 0]
    for k in ("targets", "targets_overlap"):
        ret, pcr, (lab, z, nz, counts) = got[k]
        assert tuple(ret.shape) == (0, T) and tuple(pcr.shape) == (0, T, 400) and tuple(lab.shape) == (0, T)
        assert counts.tolist() == [0, 0], k


# ---------------------------------------------------------------- coverage
KERNELS = {"vn_nstep_returns_kernel", "vn_nstep_returns_scan_kernel", "vn_backup_kernel", "vn_pixel_control_kernel<16>",
           "vn_pixel_control_list_kernel", "vn_transition_rows_kernel", "vn_gather_rows_kernel", "vn_aux_target_kernel",
           "vn_gather_f32_chw_kernel", "vn_gather_f32_chw_vec_kernel<1>", "vn_gather_f32_chw_vec_kernel<3>",
           "vn_pc_returns_kernel", "vn_rp_count_kernel", "vn_rp_scan_kernel", "vn_rp_scatter_kernel",
           "vn_replay_sample_kernel"} | {"vn_gather_leaves_f32_kernel<%d,%d>" % (k + 1, u) for k, u in enumerate(LEAF_UNROLL)}


def test_kernel_list_matches_the_source():
    """KERNELS names every __global__ instantiation of vn_rollout.cu: 16 kernels + the 6 leaf-count instantiations."""
    import os
    src = open(os.path.join(os.path.dirname(vn.build.LIB), "csrc", "vn_rollout.cu")).read()
    names = set(re.findall(r"__global__ void __launch_bounds__\([^)]*\) (vn_\w+)", src))
    assert len(KERNELS) == 22
    assert names == {re.sub(r"<.*", "", k) for k in KERNELS}


# one run per family: (case id or None, the test body, its keyword arguments, the instantiations that run must launch)
COVERAGE = [
    ("serial_n65_t128", "test_serial_returns_bit_equal", dict(time_major=False), {"vn_nstep_returns_kernel"}),
    ("scan_n37_t33", "test_scan_returns_within_bound", dict(time_major=True), {"vn_nstep_returns_scan_kernel"}),
    ("backup_d400", "test_discounted_backup_bit_equal", {}, {"vn_backup_kernel"}),
    ("pc_rgb_c3_oddcrop", "test_pixel_control_paths_bit_equal", {},
     {"vn_pixel_control_kernel<16>", "vn_transition_rows_kernel", "vn_gather_rows_kernel",
      "vn_pixel_control_list_kernel", "vn_pc_returns_kernel"}),
    ("rows_u100_n9480", "test_gather_rows_bit_equal", {}, {"vn_gather_rows_kernel"}),
    ("aux_depth_c2_small", "test_aux_targets_bit_equal", {}, {"vn_aux_target_kernel"}),
    ("f32_vec1_84", "test_float_gathers_bit_equal", {}, {"vn_gather_f32_chw_vec_kernel<1>"}),
    ("f32_vec3_small", "test_float_gathers_bit_equal", {}, {"vn_gather_f32_chw_vec_kernel<3>"}),
    ("f32_staged_off4", "test_float_gathers_bit_equal", {}, {"vn_gather_f32_chw_kernel"}),
    ("rp_n262145", "test_rp_labels_and_lists_equal", {}, {"vn_rp_count_kernel", "vn_rp_scan_kernel", "vn_rp_scatter_kernel"}),
    ("replay_L33", "test_replay_draws_equal_the_oracle", {}, {"vn_replay_sample_kernel"}),
] + [(c.id, "test_float_leaves_bit_equal", {}, {"vn_gather_leaves_f32_kernel<%d,%d>" % (len(c.p["leaves"]), c.claims["unroll"])})
     for c in LEAF_CASES]


def test_coverage_runs_name_every_instantiation():
    """The coverage runs, taken together, expect exactly the 22 instantiations, each from a case of the table."""
    ids = {c.id for c in CASES}
    assert all(cid in ids for cid, _, _, _ in COVERAGE)
    assert set().union(*(k for _, _, _, k in COVERAGE)) == KERNELS
    assert {c.id: _plan(c, B200_SMS) for c in PC_CASES}["pc_rgb_c3_oddcrop"]["table"]


@pytest.mark.gpu
@pytest.mark.parametrize("cid,body,kw,kernels", COVERAGE, ids=[c[0] for c in COVERAGE])
def test_every_kernel_instantiation_launches(cid, body, kw, kernels):
    """Each family's case (checked bit for bit or within its bound) launches the instantiations it is there for.  The
    case runs once outside the profiler (module loading, shared-memory attributes, world and table builds), then in a
    profiler schedule of one warm-up and one recorded step: CUPTI can drop the kernel records of the first moments of a
    trace (seen in a full-suite run, where some single-kernel families came back with no library kernel), and the
    warm-up step absorbs that.  Together the families launch all 22 instantiations of vn_rollout.cu."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile, schedule
    case = next(c for c in CASES if c.id == cid)
    run = globals()[body]
    run(case, **kw)
    torch.cuda.synchronize()
    recorded = []                    # the recorded step's events, handed over when its cycle ends
    with profile(activities=[ProfilerActivity.CUDA], schedule=schedule(wait=0, warmup=1, active=1),
                 on_trace_ready=lambda p: recorded.extend(e for e in p.events()
                                                          if e.device_type == torch.autograd.DeviceType.CUDA)) as prof:
        for _ in range(2):
            run(case, **kw)
            torch.cuda.synchronize()
            prof.step()
    seen = set()
    for e in recorded:
        m = re.search(r"(vn_\w+(?:<[^>(]*>)?)\(", e.name)
        if m:
            seen.add(m.group(1).replace(" ", ""))
    if not recorded:
        pytest.skip("the profiler captured no CUDA activity (CUPTI unavailable)")
    assert kernels <= seen, (sorted(kernels - seen), sorted(seen))
