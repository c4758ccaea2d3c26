"""On-disk / in-memory scene formats of the reference -> GridScene with explicit planes.

* pickled ``ThorGridWorld`` (graph/multi_graph_no_tp.py:6-25; attribute names as printed by
  testPickles.py:23-37): ``_maze [X,Y]``, ``_observations/_segmentations [X,Y,4,H,W,3]``,
  ``_depths [X,Y,4,H,W,1]`` dense over the bounding box.
* the flat h5 schema written by ``save_graph_as_h5`` (graph/util.py:222-227): ``graph [S,4]``,
  ``observation [S,H,W,C]``, ``shortest_path_distance [S,S]``.

The per-step ``cv2.resize`` of ``GraphResize`` (graph/core.py:30-57) is applied ONCE here.
"""
import numpy as np

from .scenes import GridScene


def _resize_frames(frames, hw):
    """[n, H, W, C] uint8 -> [n, h, w, C] with cv2.resize (bilinear, the GraphResize default)."""
    if tuple(frames.shape[1:3]) == tuple(hw):
        return np.ascontiguousarray(frames)
    import cv2
    out = np.empty((frames.shape[0], hw[0], hw[1], frames.shape[3]), frames.dtype)
    for i, f in enumerate(frames):
        r = cv2.resize(f, (hw[1], hw[0]))            # cv2 takes (width, height); the reference passes a square size
        out[i] = r if r.ndim == 3 else r[:, :, None]  # graph/core.py:38-39 re-adds the channel axis
    return out


def skimage_resize_restated(image, out_hw):
    """``skimage.transform.resize(image, out_hw, anti_aliasing=True)`` as THORDiscreteCachedEnv._preprocess_frame
    calls it (environments/gym_ai2thor/envs/cached.py:62-64) for a uint8 [H, W, C] frame -> float64 [h, w, C] in [0, 1].
    PARITY UNPINNED: scikit-image is not installed offline and its version is not pinned by the reference; this
    restates the published algorithm (skimage 0.15-0.19): img_as_float; when down-scaling, a Gaussian pre-filter with
    sigma = (scale - 1) / 2 per spatial axis (scipy.ndimage, mode 'mirror', truncate 4); bilinear warp (order 1) with
    source coordinate (dst + 0.5) * scale - 0.5, out-of-range taps reflected about the edge; clip to the input range."""
    from scipy import ndimage
    img = np.asarray(image).astype(np.float64) / 255.0
    if img.ndim == 2:
        img = img[:, :, None]
    H, W = img.shape[:2]
    h, w = int(out_hw[0]), int(out_hw[1])
    if (H, W) == (h, w):
        return img
    sigma = (max(0.0, (H / h - 1) / 2), max(0.0, (W / w - 1) / 2), 0.0)
    lo, hi = img.min(), img.max()
    if sigma[0] > 0 or sigma[1] > 0:
        img = ndimage.gaussian_filter(img, sigma, cval=0, mode="mirror")

    def taps(n_src, n_dst):
        c = (np.arange(n_dst, dtype=np.float64) + 0.5) * (n_src / n_dst) - 0.5
        f, ce = np.floor(c), np.ceil(c)
        reflect = lambda i: np.where(i < 0, -i - 1, np.where(i >= n_src, 2 * n_src - 1 - i, i)).astype(np.int64)
        return reflect(f), reflect(ce), c - f

    r0, r1, dr = taps(H, h)
    c0, c1, dc = taps(W, w)
    dc_ = dc[None, :, None]
    top = (1 - dc_) * img[r0][:, c0] + dc_ * img[r0][:, c1]
    bot = (1 - dc_) * img[r1][:, c0] + dc_ * img[r1][:, c1]
    dr_ = dr[:, None, None]
    return np.clip((1 - dr_) * top + dr_ * bot, lo, hi)


def _resize_frames_skimage(frames, hw):
    """[n, H, W, C] uint8 -> [n, h, w, C] uint8: skimage_resize_restated, then the float64 result is stored at uint8
    precision (rint(x * 255)) - the store holds bytes; the reference would hand the float64 frame to the model."""
    if tuple(frames.shape[1:3]) == tuple(hw):
        return np.ascontiguousarray(frames)
    out = np.empty((frames.shape[0], hw[0], hw[1], frames.shape[3]), np.uint8)
    for i, f in enumerate(frames):
        out[i] = np.clip(np.rint(skimage_resize_restated(f, hw) * 255.0), 0, 255).astype(np.uint8)
    return out


def scene_from_thor_grid_world(graph, goals, screen_size=None, planes=("rgb", "depth", "segmentation"), scene_id=0,
                               name="thor"):
    """``graph``: any object with the ThorGridWorld attributes.  Frames are compacted to free cells
    (state = free_cell_rank * 4 + rotation) and resized once to ``screen_size`` (default: stored size).
    Pass ``planes`` including ``tp_rgb`` / ``tp_depth`` / ``tp_segmentation`` for the third-person variant
    (graph/thor_graph.py), whose ``render`` returns the 6-tuple of ``obs_layout="thor6"``."""
    maze = np.asarray(graph._maze).astype(bool)
    xs, ys = np.nonzero(maze)
    src = {"rgb": graph._observations, "depth": graph._depths, "segmentation": graph._segmentations}
    for name, attr in (("tp_rgb", "_tp_observations"), ("tp_depth", "_tp_depths"), ("tp_segmentation", "_tp_segmentations")):
        if hasattr(graph, attr):                    # graph/thor_graph.py:6-13 (third-person camera of the 2nd agent)
            src[name] = getattr(graph, attr)
    hw = tuple(screen_size) if screen_size is not None else tuple(src["rgb"].shape[3:5])
    explicit = {}
    for p in planes:
        a = np.asarray(src[p])[xs, ys]                              # [cells, 4, H, W, C]
        a = a.reshape((-1,) + a.shape[2:])                          # [cells * 4, H, W, C]
        explicit[p] = _resize_frames(a, hw)
    return GridScene(maze, [tuple(g) for g in goals], True, hw, tuple(planes), scene_id=scene_id, name=name,
                     explicit=explicit)


def scene_from_h5_arrays(graph, observation, shortest_path_distance=None, location=None, goals=(), scene_id=0,
                         name="thor-h5", screen_size=None, resize="skimage"):
    """Flat h5 schema -> GridScene.  The grid geometry is recovered from the adjacency: states are
    grouped in fours (one free cell each, graph/util.py:229-237) and laid out on a single row of a
    [1, cells] maze when no ``location`` is given - the env only ever uses the flat ``graph`` table.
    ``screen_size`` other than the stored size resizes every frame ONCE here: ``resize="skimage"`` with the restated
    anti-aliased filter of THORDiscreteCachedEnv._preprocess_frame (cached.py:62-64; unpinned, see
    skimage_resize_restated), ``resize="cv2"`` with GraphResize's bilinear cv2.resize (graph/core.py:36-40)."""
    graph = np.asarray(graph)
    S = graph.shape[0]
    assert S % 4 == 0
    cells = S // 4
    obs = np.ascontiguousarray(observation)
    if screen_size is not None and tuple(screen_size) != tuple(obs.shape[1:3]):
        obs = (_resize_frames_skimage if resize == "skimage" else _resize_frames)(obs, tuple(screen_size))
    sc = GridScene(np.ones((1, cells), bool), list(goals), True, tuple(obs.shape[1:3]), ("rgb",), scene_id=scene_id,
                   name=name, explicit={"rgb": obs})
    sc.h5_graph = graph.astype(np.int32)         # used verbatim by tables.compile_world for THOR_CACHED
    # start-state candidates of a goal g are {s : shortest_path_distance[s][g] > 0} (cached.py:41-44)
    sc.h5_spd = None if shortest_path_distance is None else np.asarray(shortest_path_distance)
    return sc


def load_scene_h5(path, goals=(), screen_size=None, resize="skimage", scene_id=0):
    """Reads a scene file written by ``save_graph_as_h5`` (graph/util.py:202-247) the way
    ``THORDiscreteCachedEnv.__init__`` does (cached.py:26-32: datasets ``graph``, ``observation``,
    ``shortest_path_distance`` fully loaded with ``[()]``; ``location`` and ``resnet_feature`` are not used by the
    env) and returns the GridScene for ``compile_world([...], THOR_CACHED, tasks=[(0, goal_state), ...])``.
    h5py is an optional dependency (absent from the offline image): without it this raises ImportError naming
    ``scene_from_h5_arrays`` as the way in for arrays obtained otherwise."""
    try:
        import h5py
    except ImportError as e:        # pragma: no cover - exercised with a stand-in module in the tests
        raise ImportError("load_scene_h5 needs h5py (not installed); load the datasets 'graph', 'observation', "
                          "'shortest_path_distance' yourself and call loaders.scene_from_h5_arrays") from e
    with h5py.File(path, "r") as f:
        graph = f["graph"][()]
        observation = f["observation"][()]
        spd = f["shortest_path_distance"][()]
    return scene_from_h5_arrays(graph, observation, spd, goals=goals, scene_id=scene_id, name=str(path),
                                screen_size=screen_size, resize=resize)


# --------------------------------------------------------------------------- scene pickles without the reference tree
class _Bag:
    """Stand-in for the reference classes inside a scene pickle (graph.*.ThorGridWorld and friends are plain
    objects whose state is their ``__dict__``)."""

    def __setstate__(self, state):
        if isinstance(state, dict):
            self.__dict__.update(state)

    @property
    def maze(self):                                  # GridWorldScene.maze, graph/core.py
        return self._maze


def load_scene_pickle(path_or_file):
    """``graph.util.load_graph`` (graph/util.py:69-79) for a box that does not have the reference package: classes
    of the ``graph`` / ``environments`` packages found in the pickle are replaced by attribute bags, everything
    else (numpy arrays, tuples) unpickles normally.  Returns an object with the ThorGridWorld attributes
    (``_maze``, ``_observations``, ``_depths``, ``_segmentations``, optionally ``_tp_*``, ``goals``).  The cached
    ``graph`` / ``optimal_actions`` tables of dump_graph are ignored: tables.compile_world recomputes them (BFS)."""
    import pickle

    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            root = module.split(".")[0]
            if root in ("graph", "environments", "environment"):
                return _Bag
            return super().find_class(module, name)

    if isinstance(path_or_file, (str, bytes)) or hasattr(path_or_file, "__fspath__"):
        with open(path_or_file, "rb") as f:
            return _Unpickler(f).load()
    return _Unpickler(path_or_file).load()


#: scene name -> goals, environments/gym_graph/download.py:21-29 (the -174 variants share the goals)
THOR_CACHED_GOALS = {
    "thor-cached-212": [(3, 1, 2), (13, 21, 3), (10, 2, 1), (10, 14, 0)],
    "thor-cached-208": [(6, 3, 1), (13, 3, 0), (7, 18, 2), (6, 25, 1)],
    "thor-cached-218": [(6, 22, 1), (7, 0, 0), (18, 18, 3), (13, 31, 3)],
    "thor-cached-225": [(3, 17, 2), (12, 17, 3), (15, 10, 0), (14, 8, 3)],
}

#: gym ids of environments/gym_graph/__init__.py:8-28 -> (observation layout, max_episode_steps)
GYM_IDS = {"OrientedGraph-v0": ("frame", 900), "AuxiliaryGraph-v0": ("aux5", 900)}


def scene_file(graph_name):
    """Where the reference caches its scene pickles: ~/.visual_navigation/scenes/<name>.pkl (download.py:38-43)."""
    import os
    return os.path.join(os.path.expanduser("~"), ".visual_navigation", "scenes", "%s.pkl" % graph_name)


def make_vec(id, tasks, num_envs=None, screen_size=None, graph_files=None, **env_kwargs):
    """``create_envs`` of the experiments in one call (thor_cached_auxiliary.py:58-71): ``id`` is a gym id of
    environments/gym_graph/__init__.py ('AuxiliaryGraph-v0', 'OrientedGraph-v0', 'Graph<Scene>-v0'), ``tasks`` the
    experiment's ``[(scene_name, [goal, ...]), ...]`` list (``None`` goals = the table of download.py:21-29).  One env
    per (scene, goal) unless ``num_envs`` says otherwise; scene pickles come from ``graph_files[scene_name]`` or the
    reference's cache directory.  Returns a GraphVecEnv (extra keyword arguments, e.g. ``reward_progress``, are passed
    on)."""
    from .tables import GYM_GRAPH, compile_world
    from .vec_env import GraphVecEnv
    if id in GYM_IDS:
        layout, limit = GYM_IDS[id]
    elif id.startswith("Graph") and id.endswith("-v0"):
        layout, limit = "frame", 100                    # gym_graph/__init__.py:8-17
    else:
        raise ValueError("unknown environment id %r" % (id,))
    scenes, task_list = [], []
    for k, (name, goals) in enumerate(tasks):
        if goals is None:
            goals = THOR_CACHED_GOALS[name[:-4] if name.endswith("-174") else name]
        path = (graph_files or {}).get(name) or scene_file(name)
        graph = load_scene_pickle(path)
        planes = ("rgb", "depth", "segmentation") if layout == "aux5" else ("rgb",)
        scenes.append(scene_from_thor_grid_world(graph, goals, screen_size=screen_size, planes=planes, scene_id=k,
                                                 name=name))
        task_list += [(k, tuple(g)) for g in goals]
    world = compile_world(scenes, GYM_GRAPH, tasks=task_list)
    env_kwargs.setdefault("max_episode_steps", limit)
    env_kwargs.setdefault("obs_layout", layout)
    return GraphVecEnv(world, num_envs or len(task_list), **env_kwargs)
