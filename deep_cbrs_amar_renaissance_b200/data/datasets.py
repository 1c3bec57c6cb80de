"""Batch sequences (mirror of /root/reference/src/data/datasets.py:8-143,146-213,309-373).

They define the gather indices of the hot path: batch b of epoch e is
ratings[perm_e[b*B:(b+1)*B]] with perm_e drawn from ONE persistent
np.random.RandomState(seed) re-shuffling a fresh arange at every epoch end.
"""
import numpy as np

from .. import checkpoint


class Sequence:
    """Stand-in for keras.utils.Sequence: indexable, sized, with an epoch hook."""

    def __len__(self):
        raise NotImplementedError

    def __getitem__(self, idx):
        raise NotImplementedError

    def on_epoch_end(self):
        pass

    def get_state(self):
        """{name: ndarray}: what decides the batches of the epochs to come (the row order and the RandomState that
        reshuffles it), saved by keras_like.BackupAndRestore so that a resumed fit replays them."""
        return {}

    def set_state(self, state):
        """Put back get_state()'s arrays (ndarrays or anything np.asarray reads)."""

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class _RatingBatches(Sequence):
    def __init__(self, ratings, users, items, batch_size, shuffle, seed):
        self.ratings, self.users, self.items = ratings, users, items
        self.batch_size, self.shuffle, self.seed = batch_size, shuffle, seed
        self.indexes = None
        self.random_state = None
        self.on_epoch_end()

    def __len__(self):
        return int(np.ceil(len(self.ratings) / self.batch_size))

    def _rows(self, idx):
        lo = idx * self.batch_size
        hi = min(lo + self.batch_size, len(self.ratings))
        return self.ratings[self.indexes[lo:hi]] if self.shuffle else self.ratings[lo:hi]

    def on_epoch_end(self):
        if not self.shuffle:
            return
        if self.random_state is None:
            self.random_state = np.random.RandomState(self.seed)
        self.indexes = np.arange(len(self.ratings))
        self.random_state.shuffle(self.indexes)

    def get_state(self):
        if not self.shuffle:
            return {}
        return dict(checkpoint.rng_arrays(self.random_state), indexes=self.indexes)

    def set_state(self, state):
        if self.shuffle:
            checkpoint.set_rng(self.random_state, state)
            self.indexes = np.array(state["indexes"], dtype=np.int64)


def _sub_states(subs):
    return {name + "/" + k: a for name, seq in subs for k, a in seq.get_state().items()}


def _set_sub_states(subs, state):
    for name, seq in subs:
        seq.set_state({k[len(name) + 1:]: a for k, a in state.items() if k.startswith(name + "/")})


class UserItemGraph(_RatingBatches):
    """((user_ids, item_ids), ratings) batches + the adjacency (datasets.py:146-213)."""

    def __init__(self, ratings, users, items, adj_matrix, batch_size=512, shuffle=False, seed=42):
        self.adj_matrix = adj_matrix
        super().__init__(ratings, users, items, batch_size, shuffle, seed)

    def __getitem__(self, idx):
        r = self._rows(idx)
        return (r[:, 0], r[:, 1]), r[:, 2]


class UserItemEmbeddings(_RatingBatches):
    """((emb[user], emb[item]), ratings) batches gathered on the host (datasets.py:8-77)."""

    def __init__(self, ratings, users, items, embeddings, batch_size=512, shuffle=False, seed=42):
        self.embeddings = embeddings
        super().__init__(ratings, users, items, batch_size, shuffle, seed)

    def __getitem__(self, idx):
        r = self._rows(idx)
        return (self.embeddings[r[:, 0]], self.embeddings[r[:, 1]]), r[:, 2]


class HybridUserItemEmbeddings(Sequence):
    """((graph[user], graph[item], bert[user], bert[item]), ratings): the pre-computed-embedding hybrid baseline
    (datasets.py:80-143).  Two UserItemEmbeddings with the same seed, hence the same permutation."""

    def __init__(self, ratings, users, items, graph_embeddings, bert_embeddings, batch_size=512, shuffle=False, seed=42):
        self.ratings, self.users, self.items = ratings, users, items
        self.graph_embeddings = UserItemEmbeddings(ratings, users, items, graph_embeddings, batch_size, shuffle, seed)
        self.bert_embeddings = UserItemEmbeddings(ratings, users, items, bert_embeddings, batch_size, shuffle, seed)

    def __len__(self):
        return len(self.graph_embeddings)

    def __getitem__(self, idx):
        (ug, ig), y = self.graph_embeddings[idx]
        (ub, ib), _ = self.bert_embeddings[idx]
        return (ug, ig, ub, ib), y

    def on_epoch_end(self):
        self.graph_embeddings.on_epoch_end()
        self.bert_embeddings.on_epoch_end()

    def get_state(self):
        return _sub_states([("graph_embeddings", self.graph_embeddings), ("bert_embeddings", self.bert_embeddings)])

    def set_state(self, state):
        _set_sub_states([("graph_embeddings", self.graph_embeddings), ("bert_embeddings", self.bert_embeddings)], state)


class UserItemGraphEmbeddings(Sequence):
    """((user_ids, item_ids, bert[user], bert[item]), ratings) (datasets.py:309-373).

    Both sub-sequences own a RandomState(seed) and therefore draw the same
    permutation.  `device_resident=True` is the B200 path: the content table is
    uploaded once and only the ids travel per batch; the model gathers on
    device (HybridBertGNN accepts a 2-tuple then)."""

    def __init__(self, ratings, users, items, adj_matrix, embeddings, batch_size=512, shuffle=False,
                 seed=42, device_resident=False):
        self.ratings, self.users, self.items, self.adj_matrix = ratings, users, items, adj_matrix
        self.graph_ids = UserItemGraph(ratings, users, items, adj_matrix, batch_size, shuffle, seed)
        self.embeddings = UserItemEmbeddings(ratings, users, items, embeddings, batch_size, shuffle, seed)
        self.device_resident = device_resident

    def __len__(self):
        return len(self.graph_ids)

    def __getitem__(self, idx):
        (u, i), y = self.graph_ids[idx]
        if self.device_resident:
            return (u, i), y
        (ub, ib), _ = self.embeddings[idx]
        return (u, i, ub, ib), y

    def on_epoch_end(self):
        self.graph_ids.on_epoch_end()
        self.embeddings.on_epoch_end()

    def get_state(self):
        return _sub_states([("graph_ids", self.graph_ids), ("embeddings", self.embeddings)])

    def set_state(self, state):
        _set_sub_states([("graph_ids", self.graph_ids), ("embeddings", self.embeddings)], state)
