"""Host plumbing the recommenders share (daisyrec_b200/model/AbstractRecommender.py), checked without a device: the test
loader decode, the split of host-drawn dropout masks into calls, and the DataLoader plan of the auto-encoder models."""
import numpy as np
import pandas as pd
import pytest
import torch
from torch.utils.data import DataLoader

from daisyrec_b200.model.AbstractRecommender import candidate_rows, loader_plan, mask_segments
from daisyrec_b200.utils.dataset import AEDataset, CandidatesDataset, get_dataloader


def _rows(n=11, C=5, seed=0):
    rs = np.random.RandomState(seed)
    return [[int(u), rs.randint(0, 50, C)] for u in rs.permutation(n)]


def test_candidate_rows_list_and_iterable_agree():
    rows = _rows()
    loader = get_dataloader(CandidatesDataset(rows), batch_size=4, shuffle=False)          # 11 rows: ragged last batch
    users, cands = candidate_rows(loader)
    assert users.dtype == np.int64 and cands.dtype == np.int64 and cands.shape == (11, 5)
    assert np.array_equal(users, [r[0] for r in rows]) and np.array_equal(cands, np.stack([r[1] for r in rows]))
    batches = list(DataLoader(CandidatesDataset(rows), batch_size=4, shuffle=False))
    assert [len(b[0]) for b in batches] == [4, 4, 3]
    it_users, it_cands = candidate_rows(batches)                                            # a plain iterable of batches
    assert it_users.dtype == np.int64 and it_cands.dtype == np.int64
    assert np.array_equal(it_users, users) and np.array_equal(it_cands, cands)


@pytest.mark.parametrize("loader", [get_dataloader(CandidatesDataset([]), batch_size=4, shuffle=False), []],
                         ids=["empty-dataset", "empty-iterable"])
def test_candidate_rows_empty(loader):
    users, cands = candidate_rows(loader)
    assert users.shape == (0,) and users.dtype == np.int64 and len(cands) == 0


@pytest.mark.parametrize("n_rows,batch,first,n_steps,bytes_per_step,cap", [
    (1000, 64, 0, 16, 100, 350),          # ragged last step, three steps a call
    (1024, 64, 0, 16, 100, 350),          # exact multiple: no ragged step
    (30, 64, 0, 1, 100, 64 << 20),        # fewer rows than one batch
    (1000, 64, 5, 11, 100, 64 << 20),     # from step 5 to the end, one call plus the ragged step
    (1000, 64, 2, 4, 100, 50),            # a step's masks alone exceed the cap: one step a call
    (1000, 64, 0, 16, 100, 1600),         # the cap fits every step: the full steps, then the ragged one
    (640, 64, 0, 10, 1, 64 << 20),
])
def test_mask_segments_cover_steps_in_order(n_rows, batch, first, n_steps, bytes_per_step, cap):
    segs = list(mask_segments(n_rows, batch, first, n_steps, bytes_per_step, cap))
    assert [s + j for s, k, _ in segs for j in range(k)] == list(range(first, first + n_steps))
    for idx, (s, k, rows) in enumerate(segs):
        assert k >= 1
        if k > 1:
            assert k * bytes_per_step <= cap
        if rows != batch:                                                  # the ragged step: last, alone, the rest of the rows
            assert idx == len(segs) - 1 and k == 1 and rows == n_rows - s * batch and 0 < rows < batch
    ragged = (first + n_steps) * batch > n_rows
    assert (segs[-1][2] != batch) == ragged


def test_mask_segments_layout():
    assert list(mask_segments(1000, 64, 0, 16, 100, 350)) == [(0, 3, 64), (3, 3, 64), (6, 3, 64), (9, 3, 64), (12, 3, 64),
                                                                (15, 1, 40)]
    assert list(mask_segments(30, 64, 0, 1, 100)) == [(0, 1, 30)]
    assert list(mask_segments(1000, 64, 5, 11, 100)) == [(5, 10, 64), (15, 1, 40)]


@pytest.mark.parametrize("shuffle,drop_last", [(True, False), (False, True)])
def test_loader_plan_of_an_ae_dataset(shuffle, drop_last):
    ds = AEDataset(pd.DataFrame({"user": [3, 1, 3, 0, 2, 1], "item": [0, 1, 2, 3, 4, 5]}))
    loader = DataLoader(ds, batch_size=3, shuffle=shuffle, drop_last=drop_last)
    one_d = lambda data: data.ndim == 1  # noqa: E731
    data, bs, shuf, drop, gen = loader_plan(loader, one_d)
    assert data is ds.data and np.array_equal(data, [3, 1, 0, 2])
    assert (bs, shuf, drop, gen) == (3, shuffle, drop_last, None)
    assert loader_plan(loader) is None                                   # the default test wants [T, 3] triples
    sampler = torch.utils.data.RandomSampler(ds, generator=torch.Generator())
    assert loader_plan(DataLoader(ds, batch_size=3, sampler=sampler), one_d) is None
    assert loader_plan(list(loader), one_d) is None
