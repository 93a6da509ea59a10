"""Dataset side of the path (SURVEY §8(f) N2): the reference's JSON wire format <-> packed SoA
arrays, and the make_data.py generator (scenario sampling, instance positions, teacher rollouts
for ``ref_actions``) running on the GPU.

Wire format (data/dataset.py:39-67, make_data.py:188-216): a list of environments
``{"grid": [W][H][K] one-hot, "task_instances": [{"task": "goal[arg]", "init_pos": [[x,y]..],
"ids": ["instance_<n>"..], "ref_actions": [[a..]..]}]}``.
"""
import ctypes
import json

import numpy as np

from . import _lib
from .tables import CraftTables


# ------------------------------------------------------------------------------- wire format
def grid_to_ids(grid_onehot):
    g = np.asarray(grid_onehot)
    assert (g.sum(axis=2) <= 1).all(), "impossible world configuration"
    return (g.argmax(axis=2) * (g.sum(axis=2) > 0)).astype(np.uint8)


def ids_to_grid(ids, n_kinds):
    ids = np.asarray(ids)
    g = np.zeros(ids.shape + (n_kinds,))
    xs, ys = np.nonzero(ids)
    g[xs, ys, ids[xs, ys]] = 1
    return g


def _goal(name):
    return name if "[" in name else "%s[%s]" % tuple(name.split(" "))


def from_wire(data, tables):
    """List of env dicts (the JSON) -> dict of packed arrays: grids u8[E,W*H], inst_env,
    inst_task, inst_pos, inst_id, ref_actions (padded with 255), ref_len."""
    tm = tables.task_manager
    grids, ienv, itask, ipos, iid, acts = [], [], [], [], [], []
    for e, env in enumerate(data):
        grids.append(grid_to_ids(env["grid"]).reshape(-1))
        for ti in env["task_instances"]:
            tid = tm[_goal(ti["task"])].task_id
            for pos, id_, ra in zip(ti["init_pos"], ti["ids"], ti["ref_actions"]):
                ienv.append(e)
                itask.append(tid)
                ipos.append(pos)
                iid.append(int(str(id_).split("_")[-1]))
                acts.append(ra)
    L = max([len(a) for a in acts] + [1])
    ra = np.full((len(acts), L), 255, np.uint8)
    for i, a in enumerate(acts):
        ra[i, :len(a)] = a
    return dict(grids=np.stack(grids), inst_env=np.asarray(ienv, np.int32),
                inst_task=np.asarray(itask, np.uint8), inst_pos=np.asarray(ipos, np.uint8),
                inst_id=np.asarray(iid, np.int64), ref_actions=ra,
                ref_len=np.asarray([len(a) for a in acts], np.int32))


def to_wire(packed, tables):
    """Inverse of from_wire (instances grouped by env, then by task, in array order)."""
    tm = tables.task_manager
    W, H, K = tables.W, tables.H, tables.K
    out = []
    for e in range(len(packed["grids"])):
        item = {"grid": ids_to_grid(packed["grids"][e].reshape(W, H), K).tolist(), "task_instances": []}
        sel = np.nonzero(packed["inst_env"] == e)[0]
        by_task = {}
        for i in sel:
            by_task.setdefault(int(packed["inst_task"][i]), []).append(i)
        for tid, idxs in by_task.items():
            item["task_instances"].append({
                "task": tm.by_id(tid).goal,
                "init_pos": [packed["inst_pos"][i].tolist() for i in idxs],
                "ids": ["instance_%d" % packed["inst_id"][i] for i in idxs],
                "ref_actions": [packed["ref_actions"][i, :packed["ref_len"][i]].tolist() for i in idxs],
            })
        out.append(item)
    return out


def load_json(path, tables):
    with open(path) as f:
        return from_wire(json.load(f), tables)


def save_json(path, packed, tables):
    with open(path, "w") as f:
        json.dump(to_wire(packed, tables), f)


# ------------------------------------------------------------------------------- generation
# ------------------------------------------------------------------------------- .traj files
def eval_info(instance_ids, action_seqs, success):
    """The evaluation record the reference's trainers write as ``<split>.traj`` / ``best_dev.traj``
    (trainers/imitation.py:204-207,228-231): ``{instance id: {"actions": [...], "success": 0/1}}``.
    ``instance_ids``: ints or ``"instance_<n>"`` strings; ``action_seqs``: u8[N, L] padded with 255
    (or a list of lists); ``success``: bool[N]."""
    info = {}
    for iid, seq, ok in zip(instance_ids, action_seqs, success):
        key = iid if isinstance(iid, str) else "instance_%d" % int(iid)
        assert key not in info, key                                  # trainers/imitation.py:201
        info[key] = {"actions": [int(a) for a in seq if int(a) != 255], "success": int(bool(ok))}
    return info


def save_eval_info(path, info):
    with open(path, "w") as f:                                       # trainers/imitation.py:228-231
        json.dump(info, f)


def load_eval_info(path):
    with open(path) as f:
        return json.load(f)


def _stream(torch, device):
    return _lib.raw_stream(torch, device)


def default_placement(tables):
    """make_data.py:128-139: N_PRIMITIVES of each primitive except gold/gem (in the cookbook's
    set order), then the workshops."""
    cb = tables.cookbook
    skip = {cb.index["gold"], cb.index["gem"]}
    kinds = []
    for p in sorted(cb.primitives):
        if p in skip:
            continue
        kinds += [p] * int(tables.world_config.get("N_PRIMITIVES", 2))
    kinds += [k for k in tables.workshop_kinds]
    return np.asarray(kinds, np.uint8)


def sample_scenarios(tables, n, seed, offset=0, device=None, place_kinds=None):
    """n scenarios on the device: (scen_grid u8[n, cell_stride], init_pos u8[n,2], n_failed).
    ``place_kinds``: the kind ids to place, each in 1..K-1 (0 is the empty cell: the kernel would
    count it as occupied while the row shows it free)."""
    import torch
    pk = default_placement(tables) if place_kinds is None else np.asarray(place_kinds).reshape(-1)
    if pk.size and (pk.min() < 1 or pk.max() >= tables.K):
        raise ValueError("place_kinds must be kind ids in 1..%d, got values in %s..%s"
                         % (tables.K - 1, pk.min(), pk.max()))
    lib = _lib.load()
    ct = _lib.make_tables(tables)
    device = torch.device(device or "cuda:%d" % torch.cuda.current_device())
    cs = ((tables.W * tables.H + 63) // 64) * 64
    pk = torch.from_numpy(pk.astype(np.uint8)).to(device)
    grid = torch.empty((n, cs), dtype=torch.uint8, device=device)
    pos = torch.empty((n, 2), dtype=torch.uint8, device=device)
    fails = torch.zeros(1, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        rc = lib.psk_craft_sample_scenarios(
            ctypes.byref(ct), ctypes.c_void_p(grid.data_ptr()), ctypes.c_void_p(pos.data_ptr()),
            ctypes.c_void_p(pk.data_ptr()), len(pk), tables.cookbook.index["boundary"],
            ctypes.c_uint64(seed), ctypes.c_uint64(offset), n, cs,
            ctypes.c_void_p(fails.data_ptr()), _stream(torch, device))
    _lib.check(rc, "psk_craft_sample_scenarios")
    return grid, pos, int(fails.item())


def sample_positions(tables, scen_grid, group_scen, per_group, seed, offset=0):
    """per_group distinct random free cells for every group: u8[n_groups, per_group, 2].
    ``group_scen[g]`` is the row of ``scen_grid`` that group g draws from."""
    import torch
    gs = np.asarray(group_scen).reshape(-1)
    if gs.size and (gs.min() < 0 or gs.max() >= len(scen_grid)):
        raise ValueError("group_scen must index the %d scenario rows, got values in %s..%s"
                         % (len(scen_grid), gs.min(), gs.max()))
    lib = _lib.load()
    ct = _lib.make_tables(tables)
    device = scen_grid.device
    gs = torch.as_tensor(gs.astype(np.int32)).to(device)
    out = torch.empty((len(gs), per_group, 2), dtype=torch.uint8, device=device)
    fails = torch.zeros(1, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        rc = lib.psk_craft_sample_positions(
            ctypes.byref(ct), ctypes.c_void_p(scen_grid.data_ptr()), ctypes.c_void_p(gs.data_ptr()),
            per_group, ctypes.c_void_p(out.data_ptr()), ctypes.c_uint64(seed),
            ctypes.c_uint64(offset), len(gs), scen_grid.shape[1],
            ctypes.c_void_p(fails.data_ptr()), _stream(torch, device))
    _lib.check(rc, "psk_craft_sample_positions")
    if int(fails.item()):
        raise _lib.PskError("not enough free cells for %d positions per group" % per_group)
    return out


def generate_dataset(tables=None, n_worlds=None, n_pos=20, seed=123, max_len=64, device=None):
    """make_data.py:164-216 on the GPU: distinct scenarios, for every get/make task `n_pos`
    distinct start cells, teacher rollouts until STOP for ``ref_actions`` (each must end
    satisfied, make_data.py:151).  Returns the packed arrays of ``from_wire``."""
    import torch
    from .rollout import teacher_rollouts
    from .vec import VecCraft
    tables = tables or CraftTables()
    n_worlds = n_worlds or int(tables.world_config.get("N_WORLDS", 100))
    C = tables.W * tables.H
    # distinct grids (make_data.py:168-178): over-sample, then drop duplicates on the host
    grids, offset = [], 0
    seen = set()
    while len(grids) < n_worlds:
        g, _, fails = sample_scenarios(tables, 2 * n_worlds, seed, offset, device)
        offset += 2 * n_worlds
        if fails:
            raise _lib.PskError("scenario sampler ran out of draws")
        for row in g[:, :C].cpu().numpy():
            key = row.tobytes()
            if key not in seen and len(grids) < n_worlds:
                seen.add(key)
                grids.append(row)
    grids = np.stack(grids)
    tasks = [t.task_id for t in tables.task_manager.tasks if t.goal_name in ("get", "make")]
    n_groups = n_worlds * len(tasks)
    group_scen = np.repeat(np.arange(n_worlds, dtype=np.int32), len(tasks))
    group_task = np.tile(np.asarray(tasks, np.uint8), n_worlds)
    cs = ((C + 63) // 64) * 64
    sg = np.zeros((n_worlds, cs), np.uint8)
    sg[:, :C] = grids
    dev = torch.device(device or "cuda:%d" % torch.cuda.current_device())
    pos = sample_positions(tables, torch.from_numpy(sg).to(dev), group_scen, n_pos,
                           seed ^ 0x9E3779B97F4A7C15, 0).cpu().numpy()
    inst_env = np.repeat(group_scen, n_pos)
    inst_task = np.repeat(group_task, n_pos)
    inst_pos = pos.reshape(-1, 2)
    env = VecCraft.from_instances(tables, grids, inst_env, inst_pos, inst_task,
                                  max_timesteps=255, device=dev)
    ref, ref_len, ok = teacher_rollouts(env, max_len)
    if not bool(ok.all()):
        raise AssertionError("a teacher rollout did not end in a satisfied task")   # make_data.py:151
    return dict(grids=grids, inst_env=inst_env.astype(np.int32), inst_task=inst_task,
                inst_pos=inst_pos, inst_id=np.arange(1, len(inst_env) + 1, dtype=np.int64),
                ref_actions=ref, ref_len=ref_len)


def split_envs(packed, fractions=(0.8, 0.1, 0.1), seed=123):
    """80/10/10 split by environment (make_data.py:218-230)."""
    n_env = len(packed["grids"])
    order = np.random.RandomState(seed).permutation(n_env)
    n_train, n_dev = int(n_env * fractions[0]), int(n_env * fractions[1])
    parts = {"train": order[:n_train], "dev": order[n_train:n_train + n_dev],
             "test": order[n_train + n_dev:]}
    out = {}
    for name, envs in parts.items():
        remap = {int(e): i for i, e in enumerate(envs)}
        sel = np.nonzero(np.isin(packed["inst_env"], envs))[0]
        out[name] = dict(grids=packed["grids"][envs],
                         inst_env=np.asarray([remap[int(e)] for e in packed["inst_env"][sel]], np.int32),
                         inst_task=packed["inst_task"][sel], inst_pos=packed["inst_pos"][sel],
                         inst_id=packed["inst_id"][sel], ref_actions=packed["ref_actions"][sel],
                         ref_len=packed["ref_len"][sel])
    return out


# ------------------------------------------------------------------------------- Dataset mirror
class Dataset(object):
    """Same surface as the reference's data.Dataset (data/dataset.py:12-93): instances flattened
    to dicts {id, task, grid (one-hot ndarray), init_pos, ref_actions}, shuffled batching driven
    by ``config.random`` with the reference's call sequence (one ``shuffle`` per pass)."""

    def __init__(self, config, split, task_manager):
        import os
        self.config = config
        self.split = split
        self.task_manager = task_manager
        self.file_name = os.path.join(config.data_dir, config.world.config + "_" + split + ".json")
        with open(self.file_name) as f:
            self.data = self.flatten_data(json.load(f))
        self.instance_by_id = {item["id"]: item for item in self.data}
        self.item_idx = 0
        self.random = config.random
        self.batch_size = config.trainer.batch_size

    def __len__(self):
        return len(self.data)

    def __getitem__(self, idx):
        return self.data[idx]

    def __iter__(self):
        return iter(self.data)

    def get_instance_by_id(self, instance_id):
        return self.instance_by_id[instance_id]

    def flatten_data(self, data):
        out = []
        for env in data:
            grid = env["grid"]
            for ti in env["task_instances"]:
                task = self.task_manager[_goal(ti["task"])]
                for pos, id_, ra in zip(ti["init_pos"], ti["ids"], ti["ref_actions"]):
                    out.append({"id": id_, "task": task, "grid": np.array(grid),
                                "init_pos": tuple(pos), "ref_actions": tuple(ra)})
        return out

    def next_batch(self):
        if self.item_idx == 0:
            self.data_indices = list(range(len(self)))
            self.random.shuffle(self.data_indices)
        start, end = self.item_idx, self.item_idx + self.batch_size
        indices = self.data_indices[start:end]
        self.item_idx = end
        end_pass = self.item_idx >= len(self)
        if end_pass:
            self.item_idx = 0
        return [self[i] for i in indices], end_pass

    def iterate_batches(self):
        end_pass = False
        while not end_pass:
            batch, end_pass = self.next_batch()
            yield batch

    def packed(self, tables):
        """The same instances as the packed arrays VecCraft.from_instances takes."""
        grids, key_of, ienv, itask, ipos, acts = [], {}, [], [], [], []
        for item in self.data:
            key = item["grid"].tobytes()
            if key not in key_of:
                key_of[key] = len(grids)
                grids.append(grid_to_ids(item["grid"]).reshape(-1))
            ienv.append(key_of[key])
            itask.append(tables.task_manager[item["task"].goal_name + "[" + item["task"].goal_arg + "]"].task_id)
            ipos.append(item["init_pos"])
            acts.append(item["ref_actions"])
        L = max(len(a) for a in acts)
        ra = np.full((len(acts), L), 255, np.uint8)
        for i, a in enumerate(acts):
            ra[i, :len(a)] = a
        return dict(grids=np.stack(grids), inst_env=np.asarray(ienv, np.int32),
                    inst_task=np.asarray(itask, np.uint8), inst_pos=np.asarray(ipos, np.uint8),
                    ref_actions=ra, ref_len=np.asarray([len(a) for a in acts], np.int32))


def load(config):
    """data.load(config) of the reference (data/__init__.py): {'train','dev','test'} datasets."""
    from .tables import TaskManager
    from .worlds.craft import _given_file
    hints = getattr(getattr(config, "trainer", None), "hints", None)
    # a hint file the user named must exist (the reference's open() raises, data/task.py:36); only
    # the stock path falls back to the embedded copy when the process runs outside a checkout
    tm = TaskManager(_given_file(hints, "resources/craft/hints.hierarchy.yaml"))
    config.vocab = tm.vocab
    return {split: Dataset(config, split, tm) for split in ("train", "dev", "test")}
