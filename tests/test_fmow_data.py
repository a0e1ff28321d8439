"""fMoW partition-CSV reader + WILDS-layout image source + FedML tuple views (fedml_api/data_preprocessing/fmow/data_loader.py)."""
import os

import numpy as np
import torch

from feddrift_b200.data import fmow


def _write_partitions(root, partition="A", clients=3, steps=3):
    os.makedirs(os.path.join(root, partition))
    rng = np.random.RandomState(0)
    tables = {}
    for c in range(clients):
        for t in range(steps):
            n = [5, 1, 0, 7][(c + t) % 4]
            idx = rng.randint(0, 40, size=n)
            tables[(c, t)] = idx
            with open(fmow.partition_path(root, partition, c, t), "w") as fh:
                fh.write("\n".join(str(int(i)) for i in idx) + ("\n" if n else ""))
    return tables


def test_partition_reader_handles_single_and_empty_files(tmp_path):
    tables = _write_partitions(str(tmp_path))
    for (c, t), idx in tables.items():
        got = fmow.read_partition_indices(fmow.partition_path(str(tmp_path), "A", c, t))
        assert got.tolist() == idx.tolist()
    tabs = fmow.load_partition_tables(str(tmp_path), "A", 3, 3)
    assert len(tabs) == 3 and len(tabs[0]) == 3


def test_reference_partition_files_parse_when_present():
    # client 0 / iteration 0 of partition A, stored verbatim from the reference's data/fmow/partitions
    ref = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fmow_partitions")
    idx = fmow.read_partition_indices(fmow.partition_path(ref, "A", 0, 0))
    assert idx.ndim == 1 and len(idx) > 0 and idx.dtype == np.int64


def test_drift_data_and_fedml_views(tmp_path):
    tables = _write_partitions(str(tmp_path))
    data = fmow.fmow_drift_data(str(tmp_path), "A", train_iteration=2, num_client=3, resolution=16)
    assert data.X.shape[:2] == (3, 3) and data.X.shape[3:] == (3, 16, 16)
    src = fmow.SyntheticFmowSource(16)
    for (c, t), idx in tables.items():
        assert int(data.nsamp[t, c]) == len(idx)
        for j, i in enumerate(idx):
            assert int(data.Y[t, c, j]) == src.label(int(i))
            assert torch.equal(data.X[t, c, j], src.image(int(i)))
    C, ntr, nte, gtr, gte, local_num, tr, te, classes = fmow.load_partition_data_fmow(data, 4, 1, "win-2")
    assert C == 3 and classes == 1000 and gte is None
    for c in range(3):
        assert local_num[c] == len(tables[(c, 0)]) + len(tables[(c, 1)])
        assert sum(b[0].shape[0] for b in tr[c]) == local_num[c]
        assert sum(b[0].shape[0] for b in te[c]) == len(tables[(c, 2)])
    assert ntr == sum(local_num.values())
    allv = fmow.load_all_data_fmow(data, 4, 1)
    assert len(allv) == 3 and len(allv[0]) == 2


def test_wilds_layout_source(tmp_path):
    from PIL import Image
    root = tmp_path / "fmow_v1.1"
    (root / "images").mkdir(parents=True)
    cats = ["airport", "zoo", "barn", "airport"]
    with open(root / "rgb_metadata.csv", "w") as fh:
        fh.write("split,img_filename,category\n")
        for i, cname in enumerate(cats):
            fh.write(f"train,x{i},{cname}\n")
            Image.fromarray(np.full((8, 8, 3), 10 * (i + 1), dtype=np.uint8)).save(root / "images" / f"rgb_img_{i}.png")
    src = fmow.make_source(str(tmp_path), resolution=8)
    assert isinstance(src, fmow.WildsFmowSource)
    assert [src.label(i) for i in range(4)] == [0, 2, 1, 0]          # sorted categories: airport, barn, zoo
    x, y = src(1)
    assert x.shape == (3, 8, 8) and abs(float(x[0, 0, 0]) - 20 / 255) < 1e-6 and y == 2
