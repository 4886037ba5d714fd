"""CPU: pins oracle/dataio_port.py to the unmodified reference (its outputs on these inputs are stored in
tests/golden/dataio.npz by oracle/make_golden.py) and checks the host-side logic of nrw.raycache / nrw.mesh that needs
no GPU."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import dataio_port as dp
from oracle.make_golden import DATAIO_RANGES, DATAIO_SPLITS, dataio_getitem_inputs


@pytest.fixture(scope="module")
def G():
    return np.load(os.path.join(GOLDEN, "dataio.npz"))


@pytest.mark.parametrize("n_items,world", DATAIO_SPLITS)
def test_local_split_matches_reference(n_items, world, G):
    from nrw.raycache import local_split

    items = [f"split_{i}" for i in range(n_items)]
    for rank in range(world):
        want = [f"split_{i}" for i in G[f"split.{n_items}_{world}_{rank}"]]      # DataModule._get_local_split
        assert list(dp.local_split(items, world, rank)) == want
        assert local_split(items, world, rank) == want


def test_getitem_and_filter_match_reference(G):
    all_rays, all_rgbs, idx = dataio_getitem_inputs()
    collated = {k[len("getitem."):]: torch.from_numpy(G[k]) for k in G.files if k.startswith("getitem.")}   # PhototourismDataset.__getitem__
    got = dp.getitem_batch(all_rays, all_rgbs, idx)
    assert set(got) == set(collated)
    for k in collated:
        assert torch.equal(collated[k], got[k]), k
    assert got["rays"].shape == (97, 10) and got["ts"].dtype == torch.int64
    # the filter: lightning_modules/neuconw_system.py:345-355 executed verbatim on the collated batch
    ray_mask = torch.ones_like(collated["ts"], dtype=torch.bool)
    for name in ("person", "car", "bicycle", "minibike"):
        ray_mask[dp.LABEL_IDS[name] == collated["semantics"]] = False
    f = dp.filter_batch(got)
    assert torch.equal(f["rays"], collated["rays"][ray_mask, :]) and torch.equal(f["label"], collated["semantics"][ray_mask])
    assert 0 < f["rays"].shape[0] < 97


def test_label_ids_match_reference(G):
    m = dict(zip(G["label.names"].tolist(), G["label.ids"].tolist()))           # datasets.mask_utils.get_label_id_mapping
    for k, v in dp.LABEL_IDS.items():
        assert m[k] == v, k


@pytest.mark.parametrize("n,world", DATAIO_RANGES)
def test_local_range_matches_reference_get_local_split(n, world, G):
    from nrw.mesh import _local_range

    data = torch.arange(n * 3, dtype=torch.float32).reshape(n, 3) + 1
    for rank in range(world):
        want = torch.from_numpy(G[f"local.{n}_{world}_{rank}"])                  # utils.visualization.get_local_split
        a, b, per = dp.local_range(n, world, rank)
        assert (a, b, per) == _local_range(n, world, rank)
        assert want.shape[0] == per
        assert torch.equal(want[:max(b - a, 0)], data[a:b]) and float(want[max(b - a, 0):].abs().sum()) == 0.0


def test_sparse_lattice_dtypes_and_order():
    ind = torch.tensor([[0, 1, 2], [3, 0, 1]])
    xyz_sfm, xyz_t = dp.sparse_lattice(ind, 2, 0.125, torch.tensor([-1.0, -1.0, -1.0]), torch.tensor([0.5, 0.0, 0.0]), 2.0)
    assert xyz_sfm.dtype == torch.float32 and xyz_sfm.shape == (16, 3)
    assert torch.equal(xyz_sfm[0], torch.tensor([0 * 0.125 - 1, 2 * 0.125 - 1, 4 * 0.125 - 1]))
    assert torch.equal(xyz_sfm[1], torch.tensor([0 * 0.125 - 1, 2 * 0.125 - 1, 5 * 0.125 - 1]))     # innermost index = z
    assert torch.allclose(xyz_t, (xyz_sfm - torch.tensor([0.5, 0.0, 0.0])) / 2.0)
