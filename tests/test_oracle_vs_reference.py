"""Checks against the reference project.  The tests marked ``needs_reference`` run the UNMODIFIED reference tree
(oracle/ref_harness.py, VN_REFERENCE_ROOT) and skip where it is absent: they regenerate every golden fixture from the
reference classes and require the committed fixtures to be reproduced array for array - so the fixtures the GPU tests
replay are provably what the reference computes, not a stale or hand-edited copy.  The other tests compare with what
the reference computed as recorded in those fixtures, and run everywhere."""
import importlib.util
import os
import types

import numpy as np
import pytest

import helpers as H


def _load_generator(tmpdir):
    path = os.path.join(H.GOLDEN, "make_golden.py")
    spec = importlib.util.spec_from_file_location("make_golden_live", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.HERE = str(tmpdir)          # write the regenerated fixtures somewhere else
    return mod


@pytest.mark.needs_reference
def test_committed_goldens_reproduce_from_live_reference(tmp_path, capsys):
    from oracle import ref_harness as rh
    mg = _load_generator(tmp_path)
    ref = rh.ref_modules()
    mg.gen_graph_util(ref)
    mg.gen_gym_graph(ref)
    mg.gen_graph_env(ref)
    mg.gen_maze_render(ref)
    mg.gen_thor_cached(ref)
    mg.gen_aux_target(rh.ref_aux_trainer())
    mg.gen_trainer_contract(ref)
    mg.gen_thor_cached_tasks(ref)
    names = sorted(f for f in os.listdir(H.GOLDEN) if f.endswith(".npz"))
    assert names == sorted(f for f in os.listdir(tmp_path) if f.endswith(".npz")) and len(names) == 11
    for f in names:
        a, b = np.load(os.path.join(H.GOLDEN, f)), np.load(os.path.join(tmp_path, f))
        assert sorted(a.files) == sorted(b.files), f
        for k in a.files:
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), (f, k)


def test_reference_reset_cost_is_what_the_cpu_baseline_models():
    """The reference enumerates every free cell on EVERY reset (graph/util.py:119-143) and draws with
    ``np.random.choice(candidates, p=weights)``; tests/golden/graph_util.npz holds the weights it passed there for three
    mazes, three goals each and five complexities.  The CPU baseline's ReferenceStyleResetSource must do the same work
    on every call: the same candidate list and the same weights, and a start state drawn from that list."""
    from oracle import graph_util as gu, vec as ovec
    g = H.load("graph_util")
    for k in range(int(g["n_mazes"])):
        maze, dist, act = g["maze%d" % k], g["dist%d" % k], g["act%d" % k]
        scene = types.SimpleNamespace(maze=maze, graph=dist, optimal_actions=act)
        goals = [tuple(int(v) for v in x) for x in g["goals%d" % k]]
        maxd = int(dist.max())
        for ci, c in enumerate(g["complexities"]):
            od = None if c < 0 else c * (maxd + 4 - 1) + 1
            src = ovec.ReferenceStyleResetSource(scene, goals, lambda t, od=od: od, seed=100 * k + ci)
            calls, rng = [], src.rng
            src.rng = types.SimpleNamespace(randint=rng.randint,
                                            choice=lambda a, p=None: calls.append((len(a), p)) or rng.choice(a, p=p))
            seen = set()
            for _ in range(12):
                t, start = src()
                n, p = calls[-1]
                want = g["w_state_%d_%d_%d" % (k, t, ci)]
                assert n == len(want) and np.array_equal(p, want), (k, t, ci)
                pots, _ = gu.initial_state_candidates(maze, dist, act, goals[t])
                assert start in pots and p[pots.index(start)] > 0
                seen.add(t)
            assert len(seen) > 1


@pytest.mark.needs_reference
def test_loader_consumes_a_reference_pickle(tmp_path):
    """A scene pickled the way the reference stores them (ThorGridWorld, graph/multi_graph_no_tp.py) and read
    back with the reference's own load_graph (graph/util.py:69-79) goes through loaders.scene_from_thor_grid_world
    into the same tables / frames as the synthetic scene it was exported from."""
    import importlib
    import pickle
    from oracle import ref_harness as rh
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    T = vn.tables
    ref = rh.ref_modules()
    scene = H.scenes.make_maze_scene((9, 8), 0.2, 31, n_goals=2, planes=("rgb", "depth", "segmentation"))
    X, Y = scene.maze.shape
    arrs = {}
    for plane, c in (("rgb", 3), ("depth", 1), ("segmentation", 3)):
        a = np.zeros((X, Y, 4, 84, 84, c), np.uint8)
        a[scene.cells[:, 0], scene.cells[:, 1]] = scene.plane_frames(plane).reshape(scene.n_cells, 4, 84, 84, c)
        arrs[plane] = a
    world = ref.thor_world.ThorGridWorld(scene.maze.copy(), arrs["rgb"], arrs["depth"], arrs["segmentation"])
    world.goals = list(scene.goals)
    path = tmp_path / "scene.pkl"
    with open(path, "wb") as f:
        pickle.dump(world, f)
    graph = ref.util.load_graph(str(path))                       # adds graph.graph / graph.optimal_actions
    loaded = vn.loaders.scene_from_thor_grid_world(graph, graph.goals)
    w0, w1 = T.compile_world([scene], T.GYM_GRAPH), T.compile_world([loaded], T.GYM_GRAPH)
    assert np.array_equal(w0.adj, w1.adj) and np.array_equal(w0.cand_state, w1.cand_state)
    assert all(t.max_dist == int(np.max(graph.graph)) for t in w1.tasks)          # largest_distance, graph.py:35
    for p in ("rgb", "depth", "segmentation"):
        assert np.array_equal(loaded.plane_frames(p), scene.plane_frames(p))
    # GraphResize hoisted: what the reference would render per step at another screen size
    rz = ref.core.GraphResize(graph, (44, 44))
    small = vn.loaders.scene_from_thor_grid_world(graph, graph.goals, screen_size=(44, 44))
    for s in (0, 17, scene.n_states - 1):
        x, y, r = scene.state_tuple(s)
        rgb, depth, seg = rz.render((x, y), r, modes=["rgb", "depth", "segmentation"])
        assert np.array_equal(small.plane_frames("rgb", [s])[0], rgb)
        assert np.array_equal(small.plane_frames("depth", [s])[0], depth)
        assert np.array_equal(small.plane_frames("segmentation", [s])[0], seg)


def test_reference_trainer_accepts_the_drop_in_spaces():
    """experiments/thor_cached_auxiliary.py: ``Trainer.create_model`` (:54-56) builds the model from
    ``self.env.observation_space.spaces[0].spaces[0].shape[0]`` and ``self.env.action_space.n``.
    tests/golden/trainer_contract.npz records, from the reference's own ``Trainer`` / ``create_envs`` run unmodified,
    the arguments the Model received, the observation space it read them from and the ``set_hardness`` call
    ``create_envs`` makes (:68-70).  With the spaces of the INTEGRATION.md drop-in (GraphVecEnv's ``build_spaces``: aux5,
    scaled_float, unreal_wrapper) the Model receives the same arguments."""
    import importlib
    vn = importlib.import_module("a2cat-vn-pytorch_b200")
    vec_env = importlib.import_module("a2cat-vn-pytorch_b200.vec_env")
    g = H.load("trainer_contract")
    scene = H.trainer_contract_scene(g)
    goal = tuple(int(v) for v in g["goal"])
    assert g["unwrapped_names"][0] == "set_complexity" and g["unwrapped_calls"][0][0] == 0.01    # env.set_hardness(0.01)
    ref_leaves, ref_lar = [tuple(s) for s in g["space_leaf_shapes"].tolist()], tuple(g["space_lar_shape"].tolist())
    # the drop-in's spaces, built without a device
    w = vn.compile_world([scene], vn.GYM_GRAPH, tasks=[(0, goal)])
    obs_space, act_space = vec_env.build_spaces(w.layout, "aux5", scaled_float=True, unreal_wrapper=True)
    model_args = (obs_space.spaces[0].spaces[0].shape[0], act_space.n)                     # what create_model passes
    assert model_args == tuple(g["model_args"].tolist()) == (3, 4) and act_space.n == int(g["action_n"])
    # same nesting, same first leaf (the one the model and _get_input_for_pixel_control use, :47-48,55), same lar Box
    assert len(obs_space.spaces) == 2 and len(obs_space.spaces[0].spaces) == len(ref_leaves) == 5
    assert tuple(obs_space.spaces[0].spaces[0].shape) == ref_leaves[0] == (3, 174, 174)
    assert tuple(obs_space.spaces[1].shape) == ref_lar == (5,)
    assert obs_space.spaces[0].spaces[0].dtype == np.dtype(str(g["obs_dtypes"][0])) == np.float32
    # _get_input_for_pixel_control (:47-48) picks inputs[0][0]: the rgb leaf in both layouts
    assert vec_env.OBS_LAYOUTS["aux5"][0] == "rgb"
