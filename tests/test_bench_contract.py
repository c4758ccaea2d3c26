"""bench.py's reference arm runs without a GPU: check the one-line JSON contract (keys the driver reads), that both
arms print the same `config`, and that nothing but step launches sits inside a timed region."""
import argparse
import ast
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "1", "--port-only", "--cpu-budget", "3000"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("env-steps/s") and d["value"] > 0 and d["steps"] == 3 and d["warmup"] == 1
    assert d["config"]["workload"].startswith("C2") and d["data"] == "synthetic" and d["dtype"] == "u8"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    # best of the one-process and the N-process leg, both kept
    legs = cb["legs"]
    assert "process_1" in legs and len(legs) == 2 and d["value"] == max(l["value"] for l in legs.values())
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None
    # the SAME config object as our arm prints for the same command line (nothing measured lives in `config`)
    import bench
    args = argparse.Namespace(workload="c2", envs_per_gpu=None, hardness="none")
    assert d["config"] == bench.static_config(args, 1)
    assert d["config"]["envs_per_gpu"] == 4096 and "sample" not in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def _function_source(name):
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    node = next(n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == name)
    return ast.get_source_segment(src, node), node


def test_no_collective_inside_any_timed_region():
    """Round 1's SCALE curve measured an NCCL all-reduce that sat between the two event records.  Every timed region
    of bench.py now lives in `timed_blocks` (CUDA events) or `e2e_loop` (wall clock); neither may name a collective,
    a barrier or a synchronisation between its markers, and no other function records timing events."""
    for fn in ("timed_blocks", "e2e_loop"):
        text, node = _function_source(fn)
        body = text.split("# >>> timed region")[1].split("# <<< timed region")[0]
        for word in ("dist.", "barrier", "all_reduce", "broadcast", "all_gather", "max_over_ranks", "torch.tensor",
                     "empty(", "zeros("):
            assert word not in body, (fn, word)
        # nothing in the whole function touches torch.distributed
        names = {n.id for n in ast.walk(node) if isinstance(n, ast.Name)} | \
                {n.attr for n in ast.walk(node) if isinstance(n, ast.Attribute)}
        assert not names & {"dist", "all_reduce", "barrier", "all_gather", "broadcast"}, (fn, names)
    # the e2e loop may synchronise the DEVICE inside its window (that is part of an end-to-end step), never the ranks
    text, _ = _function_source("e2e_loop")
    assert "sync()" in text
    # the headline and every secondary device-resident leg go through Harness.blocks -> timed_blocks
    run_cuda, node = _function_source("run_cuda")
    calls = [n for n in ast.walk(node) if isinstance(n, ast.Call) and isinstance(n.func, ast.Attribute)]
    recorders = [c for c in calls if c.func.attr == "record"]
    # only the isolated per-launch gather timing, the same-size copy calibration and the stand-alone collective timing
    # record events themselves; none of them is a reported step time
    assert len(recorders) <= 8
    assert "H.blocks(lambda r: device_loop" in run_cuda


def test_timed_blocks_under_gloo_world_size_2(tmp_path):
    """World-size-2 gloo run of the timing harness with collectives that RAISE while a region is open: barriers and
    the max-over-ranks reduction happen strictly outside the event pairs, and both ranks agree on the block count."""
    script = tmp_path / "run.py"
    script.write_text(textwrap.dedent("""
        import os, sys, time
        sys.path.insert(0, %r)
        import numpy as np
        import torch, torch.distributed as dist
        import bench

        rank = int(os.environ["RANK"])
        dist.init_process_group("gloo", rank=rank, world_size=2)
        state = {"open": 0, "collectives": 0}

        class Ev:
            def record(self):
                state["open"] ^= 1
                self.t = time.perf_counter()
            def elapsed_time(self, other):
                return 1e3 * (other.t - self.t)

        class Guard:
            ReduceOp = dist.ReduceOp
            def barrier(self):
                assert not state["open"], "barrier inside a timed region"
                state["collectives"] += 1
                dist.barrier()
            def all_reduce(self, t, op=dist.ReduceOp.SUM):
                assert not state["open"], "all_reduce inside a timed region"
                state["collectives"] += 1
                dist.all_reduce(t, op=op)

        class FakeCuda:
            @staticmethod
            def synchronize(dev=None):
                assert not state["open"], "device synchronisation inside a timed region"
            @staticmethod
            def Event(enable_timing=True):
                return Ev()

        class FakeTorch:
            cuda = FakeCuda
            float64 = torch.float64
            @staticmethod
            def tensor(v, device=None, dtype=None):
                return torch.tensor(v, dtype=dtype)

        H = bench.Harness(FakeTorch, Guard(), None, 2)
        steps = []
        def run_block(r):
            assert state["open"] == 1
            time.sleep(0.001 * (1 + rank))          # rank 1 is slower: the max over ranks must pick it up
            steps.append(r)
        ms = H.blocks(run_block, 5)
        assert len(ms) == 5 and steps == list(range(5)) and state["open"] == 0
        assert all(m >= 1.9 for m in ms), ms            # rank 1's 2 ms, seen by both ranks
        nb = H.n_blocks_for(0.5 if rank == 0 else 2.0)  # ranks estimate differently, agree on the max
        assert nb == int(np.ceil(bench.MIN_REGION_S * 1e3 / 0.5)), nb
        assert state["collectives"] >= 4
        dist.barrier()
        print("OK", rank)
    """ % ROOT))
    procs = []
    port = 29500 + os.getpid() % 2000
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                                      text=True))
    for r, p in enumerate(procs):
        out, err = p.communicate(timeout=180)
        assert p.returncode == 0 and "OK %d" % r in out, err[-3000:]


def test_dump_outputs_types_budget_and_fixed_row_sample(tmp_path):
    """--dump-outputs' writer: float32 / float64 files only, integers kept exact, and arrays too large for the budget
    reduced to the same seeded rows in every array named as sampled (the others written whole)."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    obs = torch.randint(0, 256, (64, 5, 5, 3), dtype=torch.uint8, generator=g)
    arrays = [("obs", obs), ("v64", torch.rand(64, dtype=torch.float64, generator=g)),
              ("reward", torch.rand(64, generator=g)), ("done", torch.rand(64, generator=g) < 0.5),
              ("big", torch.arange(64) + (1 << 30)), ("lists", torch.arange(10, dtype=torch.int32))]
    sampled = ["obs", "v64"]
    bench.dump_outputs(str(tmp_path / "all"), arrays, sampled)
    a = {k: np.load(tmp_path / "all" / (k + ".npy")) for k, _ in arrays}
    assert a["obs"].dtype == np.float32 and np.array_equal(a["obs"], obs.numpy().astype(np.float32))
    assert a["reward"].dtype == np.float32 and a["done"].dtype == np.float32 and a["v64"].dtype == np.float64
    assert a["big"].dtype == np.float64 and np.array_equal(a["big"], np.arange(64) + (1 << 30))    # > 2^24: float64
    assert a["lists"].dtype == np.float32 and np.array_equal(a["lists"], np.arange(10))
    budget = 20 * (75 * 4 + 8) + 64 * (4 + 4 + 8) + 10 * 4
    for d in ("s0", "s1"):
        bench.dump_outputs(str(tmp_path / d), arrays, sampled, budget=budget)
    s = {k: np.load(tmp_path / "s0" / (k + ".npy")) for k, _ in arrays}
    assert all(np.array_equal(s[k], np.load(tmp_path / "s1" / (k + ".npy"))) for k in s)
    rows = np.flatnonzero((a["obs"][:, None] == s["obs"][None]).all(axis=(2, 3, 4)).any(axis=1))
    assert len(rows) == s["obs"].shape[0] == 20 and np.array_equal(s["v64"], a["v64"][rows])
    assert all(np.array_equal(s[k], a[k]) for k in ("reward", "done", "big", "lists"))
    assert sum(v.nbytes for v in s.values()) <= budget
