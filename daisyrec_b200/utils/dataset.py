"""Train / test feed objects with the reference's names (daisy/utils/dataset.py:5-38).

``BasicDataset`` and ``CandidatesDataset`` stay ordinary ``torch.utils.data.Dataset`` objects so
that drivers written for daisyRec (run_examples/test.py:93-94,118-119) work unchanged; the
B200 models do not iterate them sample by sample -- ``fit``/``rank`` read ``.data`` in bulk.
"""
import torch
from torch.utils.data import DataLoader, Dataset


def get_dataloader(ds, batch_size, shuffle, num_workers=4):
    # num_workers is accepted for source compatibility (test.py:94); the device path never forks
    # workers because it never calls __getitem__.
    return DataLoader(ds, batch_size=batch_size, shuffle=shuffle, num_workers=0 if _bulk(ds) else num_workers)


def _bulk(ds):
    return isinstance(ds, (BasicDataset, CandidatesDataset, AEDataset))


class BasicDataset(Dataset):
    """<u, i, j> rows produced by the sampler (daisy/utils/dataset.py:10-27)."""

    def __init__(self, samples):
        super().__init__()
        self.data = samples

    def __len__(self):
        return len(self.data)

    def __getitem__(self, index):
        row = self.data[index]
        return row[0], row[1], row[2]


class CandidatesDataset(Dataset):
    """[user, candidate-id array] pairs from build_candidates_set (daisy/utils/dataset.py:29-38)."""

    def __init__(self, ucands):
        super().__init__()
        self.data = ucands

    def __len__(self):
        return len(self.data)

    def __getitem__(self, index):
        u, c = self.data[index]
        return torch.tensor(u), torch.tensor(c)


class AEDataset(Dataset):
    """The users (or items) of the train set for the auto-encoder models (daisy/utils/dataset.py:40-58): ``data`` is the
    1-D array of ``train_set[yield_col].unique()``, in order of first appearance."""

    def __init__(self, train_set, yield_col='user'):
        super().__init__()
        self.data = train_set[yield_col].unique()

    def __len__(self):
        return len(self.data)

    def __getitem__(self, index):
        return self.data[index]
