"""The HBM-resident world: frame store + transition / reset tables on one GPU.

Replaces the in-RAM numpy arrays of ``ThorGridWorld`` (graph/multi_graph_no_tp.py:6-25) and the h5
datasets loaded by ``THORDiscreteCachedEnv.__init__`` (environments/gym_ai2thor/envs/cached.py:26-32).
The store is replicated per GPU (SURVEY.md section 8(e)); a 30-scene world is < 9 GB of 180 GB.

Layout: one record per (global) state, ``state_pitch`` bytes, holding every plane at a 128-byte
aligned offset (tables.StoreLayout) - the planes of one state share DRAM pages, and every gather
source is 128-byte aligned.
"""
import ctypes as C

import numpy as np
import torch

from . import lib as L
from .scenes import PLANE_ID
from .tables import World


class DeviceWorld:
    def __init__(self, world: World, device="cuda", fill=True):
        if not torch.cuda.is_available():
            raise L.VnError("a CUDA device is required: the env path has no CPU fallback")
        self.lib = L.load()
        self.world = world
        self.device = torch.device(device)
        lay = world.layout
        n = world.n_states
        with torch.cuda.device(self.device):
            self.frames = torch.empty((n, lay.state_pitch), dtype=torch.uint8, device=self.device)
            dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(self.device)
            self.adj = dev(world.adj, np.int32)
            self.task_goal = dev(world.task_goal, np.int32)
            self.task_cand_off = dev(world.task_cand_off, np.int32)
            self.cand_state = dev(world.cand_state, np.int32)
            self.task_prefix = dev(world.prefixes(None), np.int32)
        assert self.frames.data_ptr() % 128 == 0
        self.store = L.Store()
        self.store.base = self.frames.data_ptr()
        self.store.state_pitch = lay.state_pitch
        self.store.n_states = n
        self.store.n_planes = len(lay.planes)
        for i, (o, b) in enumerate(zip(lay.plane_off, lay.plane_bytes)):
            self.store.plane_off[i] = o
            self.store.plane_bytes[i] = b
        self.tables = L.Tables()
        self.tables.adj = self.adj.data_ptr()
        self.tables.task_goal = self.task_goal.data_ptr()
        self.tables.task_cand_off = self.task_cand_off.data_ptr()
        self.tables.task_prefix = self.task_prefix.data_ptr()
        self.tables.cand_state = self.cand_state.data_ptr()
        self.tables.n_states = n
        self.tables.n_tasks = len(world.tasks)
        self.complexity = None
        self._shortest = None
        if fill:
            self.fill()

    # ------------------------------------------------------------------ store build
    def fill(self):
        """Synthetic scenes: hash-fill on the device (no host copy of the frames exists).
        Scenes with explicit planes are uploaded."""
        lay = self.world.layout
        ids = (C.c_int32 * L.VN_MAX_PLANES)(*([PLANE_ID[p] for p in lay.planes] + [0] * (L.VN_MAX_PLANES - len(lay.planes))))
        with torch.cuda.device(self.device):
            for si, sc in enumerate(self.world.scenes):
                r0 = int(self.world.scene_base[si])
                if sc.explicit is not None:
                    self.upload_scene(si, sc.explicit)
                else:
                    L.check(self.lib.vn_fill_store(C.byref(self.store), r0, sc.n_states, C.c_uint64(sc.frame_seed),
                                                   sc.scene_id, 0, ids, L.current_stream()))

    def upload_scene(self, scene_index, planes):
        """planes: {name: uint8 [n_states, H, W, C]} (e.g. loaded from a scene pickle / h5 file)."""
        lay = self.world.layout
        sc = self.world.scenes[scene_index]
        r0 = int(self.world.scene_base[scene_index])
        for name, off, nb in zip(lay.planes, lay.plane_off, lay.frame_bytes):
            a = np.ascontiguousarray(planes[name]).reshape(sc.n_states, nb)
            self.frames[r0:r0 + sc.n_states, off:off + nb] = torch.from_numpy(a).to(self.device)
        pad = torch.ones(lay.state_pitch, dtype=torch.bool)
        for off, nb in zip(lay.plane_off, lay.frame_bytes):
            pad[off:off + nb] = False
        if pad.any():
            self.frames[r0:r0 + sc.n_states][:, pad.to(self.device)] = 0

    def set_complexity(self, complexity):
        """set_complexity(c) (gym_graph/graph.py:43-44): the curriculum becomes a prefix length per task."""
        self.complexity = complexity
        pre = torch.from_numpy(self.world.prefixes(complexity))
        self.task_prefix.copy_(pre.to(self.device), non_blocking=False)

    def shortest_paths(self):
        """(action, dist) int32 CUDA tensors ``[n_tasks, n_states]``: for every task and GLOBAL state the first action of
        a shortest action sequence to the task's goal and its length, -1 where the goal cannot be reached (and for the
        states of other scenes) - tables.optimal_policy_table on the state graph, orientation included.  Built on the host
        the first time it is asked for, then kept: ``n_tasks * n_states * 4`` bytes of device memory each (C2: 96 KB,
        C4's 30 scenes: 86.4 MB).  ``dist`` is also the table the step kernel reads for the geodesic-progress reward
        (vn_tables_t.task_dist), so GraphVecEnv.optimal_actions() and the reward share one copy."""
        if self._shortest is None:
            from .tables import optimal_policy_table
            w = self.world
            act = np.full((len(w.tasks), w.n_states), -1, np.int32)
            dst = np.full((len(w.tasks), w.n_states), -1, np.int32)
            for ti, t in enumerate(w.tasks):
                b = int(w.scene_base[t.scene])
                d, a = optimal_policy_table(w, ti)
                act[ti, b:b + len(a)] = a
                dst[ti, b:b + len(d)] = d
            with torch.cuda.device(self.device):
                self._shortest = (torch.from_numpy(act).to(self.device), torch.from_numpy(dst).to(self.device))
            self.tables.task_dist = self._shortest[1].data_ptr()
        return self._shortest

    def plane_index(self, name):
        return self.world.layout.planes.index(name)

    def plane_view(self, name):
        """uint8 [n_states, H, W, C] strided view of one plane inside the store."""
        lay = self.world.layout
        i = self.plane_index(name)
        h, w = lay.frame_hw
        return self.frames[:, lay.plane_off[i]:lay.plane_off[i] + lay.frame_bytes[i]].view(-1, h, w, lay.channels[i])

    def nbytes(self):
        return self.frames.numel()
