"""Dataset wire format (data/dataset.py:39-67) <-> packed arrays; CPU only."""
import numpy as np
import pytest


def test_wire_format_reads_reference_goldens(splits, medium_tables):
    """The shipped dev split, re-serialised to the reference's JSON layout and read back."""
    from psketch_b200 import data
    packed = {k[4:]: splits[k] for k in splits.files if k.startswith("dev_")}
    packed["inst_env"] = packed["inst_env"].astype(np.int32)
    packed["ref_len"] = packed["ref_len"].astype(np.int32)
    wire = data.to_wire(packed, medium_tables)
    assert len(wire) == 10 and len(wire[0]["task_instances"]) == 11
    assert np.asarray(wire[0]["grid"]).shape == (8, 8, 21)
    assert wire[0]["task_instances"][0]["task"] == "get[wood]"
    back = data.from_wire(wire, medium_tables)
    assert np.array_equal(back["grids"], packed["grids"])
    assert np.array_equal(back["ref_actions"], packed["ref_actions"])


def test_wire_format_accepts_both_task_spellings(medium_tables):
    """Shipped files say "get[wood]"; a current make_data.py writes "get wood" (data/task.py:28-29)."""
    from psketch_b200 import data
    grid = np.zeros((8, 8, 21))
    grid[0, :, 1] = grid[7, :, 1] = grid[:, 0, 1] = grid[:, 7, 1] = 1
    grid[3, 3, 9] = 1
    env = {"grid": grid.tolist(), "task_instances": [
        {"task": "get[wood]", "init_pos": [[1, 1]], "ids": ["instance_1"], "ref_actions": [[1, 5]]},
        {"task": "make plank", "init_pos": [[2, 2]], "ids": ["instance_2"], "ref_actions": [[3, 4, 5]]}]}
    p = data.from_wire([env], medium_tables)
    assert p["inst_task"].tolist() == [13, 19] and p["ref_len"].tolist() == [2, 3]
    assert p["grids"][0].reshape(8, 8)[3, 3] == 9 and p["ref_actions"][0].tolist() == [1, 5, 255]


def test_dataset_mirror_batches_like_the_reference(splits, medium_tables, tmp_path):
    """Dataset (data/dataset.py:12-93): same flattening, and the same shuffled batch order as the
    reference's own Dataset — the 30 training batches its ImitationTrainer drew with RandomState(123),
    as recorded in tests/golden/config4_imitation.npz."""
    import json
    import os
    import types
    from psketch_b200 import data

    def write(split):
        packed = {k[len(split) + 1:]: splits[k] for k in splits.files if k.startswith(split + "_")}
        packed["inst_env"] = packed["inst_env"].astype(np.int32)
        packed["ref_len"] = packed["ref_len"].astype(np.int32)
        json.dump(data.to_wire(packed, medium_tables), open(str(tmp_path / ("craft_medium_%s.json" % split)), "w"))
        return packed
    packed = write("dev")
    write("train")

    def cfg(seed):
        return types.SimpleNamespace(data_dir=str(tmp_path), world=types.SimpleNamespace(config="craft_medium"),
                                     trainer=types.SimpleNamespace(batch_size=32, hints=None),
                                     random=np.random.RandomState(seed))
    ds = data.Dataset(cfg(3), "dev", medium_tables.task_manager)
    assert len(ds) == 2200 and ds[0]["grid"].shape == (8, 8, 21) and ds[0]["task"].goal_name == "get"
    assert ds.get_instance_by_id(ds[5]["id"]) is ds[5]
    batches = list(ds.iterate_batches())
    assert len(batches) == 69 and len(batches[-1]) == 2200 - 68 * 32
    back = ds.packed(medium_tables)
    assert np.array_equal(back["inst_pos"], packed["inst_pos"]) and np.array_equal(back["ref_actions"], packed["ref_actions"])
    rec = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config4_imitation.npz"))
    train = data.Dataset(cfg(123), "train", medium_tables.task_manager)
    row = {it["id"]: i for i, it in enumerate(train.data)}
    batches = train.iterate_batches()
    for r in range(int(rec["n_train_iters"])):
        got = [row[it["id"]] for it in next(batches)]
        assert got == rec["batch"][r, :int(rec["n_env"][r])].tolist(), r


def test_traj_files_have_the_reference_format(tmp_path):
    """trainers/imitation.py:204-207,228-231: {instance id: {'actions': [...], 'success': 0/1}}."""
    import json
    from psketch_b200 import data
    acts = np.asarray([[3, 3, 4, 5, 255, 255], [0, 5, 255, 255, 255, 255], [1, 1, 1, 1, 1, 1]], np.uint8)
    info = data.eval_info([10561, "instance_7", 3], acts, [True, False, True])
    assert info == {"instance_10561": {"actions": [3, 3, 4, 5], "success": 1},
                    "instance_7": {"actions": [0, 5], "success": 0},
                    "instance_3": {"actions": [1, 1, 1, 1, 1, 1], "success": 1}}
    path = str(tmp_path / "dev.traj")
    data.save_eval_info(path, info)
    assert json.load(open(path)) == info == data.load_eval_info(path)
    with pytest.raises(AssertionError):
        data.eval_info([1, 1], acts[:2], [True, True])
