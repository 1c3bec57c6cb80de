"""Weight files, optimiser state and training backups on the host (deep_cbrs_amar_renaissance_b200/checkpoint.py,
keras_like.Model.save_weights / load_weights / BackupAndRestore, training.Adam.state_dict / load_state_dict): the
round trip of names, shapes and dtypes; every refusal happens before anything is written and names the offending
path; files load without pickle; a leftover temporary file of an interrupted write is ignored."""
import os
import zipfile

import numpy as np
import pytest
import torch

from deep_cbrs_amar_renaissance_b200 import checkpoint
from tests.test_host_logic_cpu import shape_only_graphs  # noqa: F401  (fixture)

HYB_UNITS = [[16, 16], [16, 8], [16, 16]]


def _models(name):
    """a built model of `name` and a fresh, unbuilt one with another seed"""
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic, hybrid
    from tests.helpers import random_bipartite
    adj = random_bipartite(30, 20, 200, seed=1)
    out = []
    for seed in (1, 2):
        set_seed(seed)
        if name == "BasicGCN":
            m = basic.BasicGCN(adj, n_hiddens=[8, 8], embedding_dim=8, dense_units=[16, 8], clf_units=[8, 8])
        elif name == "HybridBertGAT":
            m = hybrid.HybridBertGAT(adj, n_hiddens=[8, 8], embedding_dim=8, dense_units=HYB_UNITS, clf_units=[16, 16],
                                     feature_based=True)
        elif name == "BasicRS":
            m = basic.BasicRS(dense_units=[16, 8], clf_units=[8])
        else:
            m = hybrid.HybridCBRS(feature_based=False, dense_units=HYB_UNITS, clf_units=[16, 16],
                                  fusion_method="attention")
        if seed == 1:
            {"BasicGCN": lambda: m.build_weights(), "HybridBertGAT": lambda: m.build_weights(12),
             "BasicRS": lambda: m.build_for(10), "HybridCBRS": lambda: m.build_for(10, 12)}[name]()
        out.append(m)
    return out


def _snapshot(model):
    return [(n, w.detach().cpu().clone()) for n, w in model.named_weights()]


def _same(a, b):
    return [n for n, _ in a] == [n for n, _ in b] and all(torch.equal(x, y) for (_, x), (_, y) in zip(a, b))


@pytest.mark.parametrize("name", ["BasicGCN", "HybridBertGAT", "BasicRS", "HybridCBRS"])
def test_weights_round_trip_by_path_into_an_unbuilt_model(shape_only_graphs, tmp_path, name):  # noqa: F811
    src, dst = _models(name)
    assert dst.count_params() < src.count_params()          # not built yet (the GNNs hold only their table)
    path = str(tmp_path / "w.npz")
    src.save_weights(path)
    dst.load_weights(path)
    assert _same(_snapshot(dst), _snapshot(src))
    assert all(w.dtype == torch.float32 for w in dst.weights)
    with np.load(path, allow_pickle=False) as f:            # plain numpy, no code runs on load
        header = f["header"].tobytes().decode()
        assert set(f.files) == {"header"} | {n for n, _ in src.named_weights()}
        for n, w in src.named_weights():
            assert f[n].dtype == np.float32 and f[n].shape == tuple(w.shape)
    assert name in header and '"kind": "weights"' in header
    if name == "BasicGCN":
        assert "gnn/gnn_layers/seq_layers.0/kernel" in header and "rs/clf/layers.2/bias" in header


def _rewrite(src_path, dst_path, change):
    """copy of a weight file with its arrays (and the header's list) changed by change(dict) -> dict"""
    with checkpoint.Reader(src_path, "weights") as rd:
        arrays = {k: np.asarray(v) for k, v in rd.arrays().items()}
        header = dict(rd.header)
    arrays = change(arrays)
    header["weights"] = checkpoint.spec(arrays.items())
    checkpoint.write(dst_path, header, list(arrays.items()))


def _drop(k):
    def f(a):
        del a[k]
        return a
    return f


def _set(k, v):
    def f(a):
        a[k] = v
        return a
    return f


@pytest.mark.parametrize("case", ["missing", "extra", "shape", "dtype", "class"])
def test_a_bad_weight_file_is_refused_before_any_write(shape_only_graphs, tmp_path, case):  # noqa: F811
    src, dst = _models("BasicGCN")
    dst.build_weights()
    path, bad = str(tmp_path / "w.npz"), str(tmp_path / "bad.npz")
    src.save_weights(path)
    k = "gnn/gnn_layers/seq_layers.1/kernel"
    kern = dict(src.named_weights())[k].detach().cpu().numpy()
    change = {"missing": _drop(k), "extra": _set("rs/clf/layers.9/bias", np.zeros(3, np.float32)),
              "shape": _set(k, kern[:, :-1].copy()), "dtype": _set(k, kern.astype(np.float64)),
              "class": lambda a: a}[case]
    _rewrite(path, bad, change)
    if case == "class":
        _, other = _models("HybridBertGAT")
        other.build_weights(12)
        before = _snapshot(other)
        with pytest.raises(ValueError, match="BasicGCN"):
            other.load_weights(bad)
        assert _same(_snapshot(other), before)
        return
    before = _snapshot(dst)
    with pytest.raises(ValueError, match=("rs/clf/layers.9/bias" if case == "extra" else k)):
        dst.load_weights(bad)
    assert _same(_snapshot(dst), before)


def test_an_array_that_needs_pickle_is_refused(shape_only_graphs, tmp_path):  # noqa: F811
    src, dst = _models("BasicRS")
    path = str(tmp_path / "w.npz")
    src.save_weights(path)
    with checkpoint.Reader(path, "weights") as rd:
        arrays = {k: np.asarray(v) for k, v in rd.arrays().items()}
        header = rd.header
    arrays["unet/layers.0/kernel"] = np.array([object()], dtype=object)
    with zipfile.ZipFile(path, "w") as zf:                 # np.savez would pickle the object array
        for name, a in [("header", np.frombuffer(__import__("json").dumps(header).encode(), np.uint8))] + list(arrays.items()):
            with zf.open(name + ".npy", "w") as f:
                np.lib.format.write_array(f, a, allow_pickle=True)
    with pytest.raises(ValueError, match="unet/layers.0/kernel"):
        dst.load_weights(path)


def _adam_state(model, adam, seed):
    g = torch.Generator().manual_seed(seed)
    for w in model.weights[:4]:
        adam._state[id(w)] = (torch.rand(w.shape, generator=g).to(w.device), torch.rand(w.shape, generator=g).to(w.device))
    adam.iterations = 7


def test_adam_state_round_trip_and_refusals(shape_only_graphs):  # noqa: F811
    from deep_cbrs_amar_renaissance_b200.training import Adam
    src, dst = _models("BasicGCN")
    dst.build_weights()
    a = Adam(learning_rate=1e-2)
    _adam_state(src, a, 0)
    st = a.state_dict(src)
    paths = [n for n, _ in src.named_weights()][:4]
    assert st["iterations"] == 7 and st["learning_rate"] == 1e-2 and list(st["m"]) == paths == list(st["v"])
    b = Adam(learning_rate=1e-2)
    _adam_state(dst, b, 1)                                 # existing slots are filled in place
    slots = {id(w): b._state[id(w)] for w in dst.weights[:4]}
    b.load_state_dict(dst, {k: (v if k not in "mv" else {p: t.cpu().numpy() for p, t in v.items()})
                            for k, v in st.items()})
    assert b.iterations == 7
    for p, w in zip(paths, dst.weights[:4]):
        assert b._state[id(w)] is slots[id(w)]
        assert torch.equal(b._state[id(w)][0].cpu(), st["m"][p].cpu()) and torch.equal(b._state[id(w)][1].cpu(), st["v"][p].cpu())
    fresh = Adam(learning_rate=1e-2)
    fresh.load_state_dict(dst, st)                         # no slots yet: created
    assert sorted(fresh._state) == sorted(id(w) for w in dst.weights[:4])

    def unchanged(opt, call, match):
        before = {k: (m.clone(), v.clone()) for k, (m, v) in opt._state.items()}
        it = opt.iterations
        with pytest.raises(ValueError, match=match):
            call()
        assert opt.iterations == it and sorted(opt._state) == sorted(before)
        assert all(torch.equal(opt._state[k][0], m) and torch.equal(opt._state[k][1], v) for k, (m, v) in before.items())

    for k, v in (("learning_rate", 1e-3), ("beta_1", 0.8), ("beta_2", 0.99), ("epsilon", 1e-8)):
        unchanged(b, lambda: b.load_state_dict(dst, dict(st, **{k: v})), k)
    p0 = paths[1]
    bad_shape = dict(st, m=dict(st["m"], **{p0: st["m"][p0][:1]}))
    unchanged(b, lambda: b.load_state_dict(dst, bad_shape), p0)
    bad_dtype = dict(st, v=dict(st["v"], **{p0: st["v"][p0].double()}))
    unchanged(b, lambda: b.load_state_dict(dst, bad_dtype), p0)
    unchanged(b, lambda: b.load_state_dict(dst, dict(st, m=dict(st["m"], nope=st["m"][p0]))), "nope")
    only_m = dict(st, v={p: t for p, t in st["v"].items() if p != p0})
    unchanged(b, lambda: b.load_state_dict(dst, only_m), p0)


def test_sequence_state_replays_the_coming_epochs():
    from deep_cbrs_amar_renaissance_b200.data.datasets import UserItemGraphEmbeddings
    rng = np.random.RandomState(0)
    ratings = np.stack([rng.randint(0, 30, 500), rng.randint(30, 50, 500), rng.randint(0, 2, 500)], axis=1)
    emb = rng.standard_normal((50, 4)).astype(np.float32)
    make = lambda: UserItemGraphEmbeddings(ratings, np.arange(30), np.arange(20), None, emb, batch_size=64,  # noqa: E731
                                           shuffle=True, seed=3)
    a = make()
    a.on_epoch_end()
    st = a.get_state()
    assert set(st) == {"graph_ids/indexes", "graph_ids/rng_keys", "graph_ids/rng_tail", "embeddings/indexes",
                       "embeddings/rng_keys", "embeddings/rng_tail"}
    b = make()
    b.set_state({k: v.copy() for k, v in st.items()})
    for _ in range(3):
        for k in range(len(a)):
            (xa, ya), (xb, yb) = a[k], b[k]
            assert all(np.array_equal(p, q) for p, q in zip(xa, xb)) and np.array_equal(ya, yb)
        a.on_epoch_end()
        b.on_epoch_end()


class _Seq:
    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


def test_backup_is_atomic_and_a_leftover_temporary_file_is_ignored(shape_only_graphs, tmp_path):  # noqa: F811
    from deep_cbrs_amar_renaissance_b200.keras_like import BackupAndRestore, History, _FitState
    src, dst = _models("BasicRS")
    src.compile(optimizer={"learning_rate": 1e-2})
    _adam_state(src, src.adam(), 3)
    folder = tmp_path / "backup"

    def fit_state(model, epoch):
        h = History()
        if epoch:
            h.history, h.epoch = {"loss": [0.5, 0.25]}, [0, 1]
        rng = np.random.RandomState(model.shuffle_seed)
        for _ in range(epoch):
            rng.permutation(4)
        model._fit_state = _FitState(_Seq(4), rng, h, epoch)
        return model._fit_state

    cb = BackupAndRestore(str(folder))
    cb.set_model(src)
    st_src = fit_state(src, 2)
    cb.on_epoch_end(1)
    assert sorted(os.listdir(folder)) == [BackupAndRestore.FILE]
    # a write that dies midway leaves the previous file and no temporary file
    with pytest.raises(RuntimeError):
        checkpoint.write(str(folder / BackupAndRestore.FILE), {},
                         (("x", np.zeros(1)) if k == 0 else (_ for _ in ()).throw(RuntimeError("killed"))
                          for k in range(2)))
    assert sorted(os.listdir(folder)) == [BackupAndRestore.FILE]
    # the leftover of a write killed before its rename
    (folder / ("." + BackupAndRestore.FILE + ".abc123.tmp")).write_bytes(b"PK\x03\x04 torn")
    dst.compile(optimizer={"learning_rate": 1e-2})
    cb2 = BackupAndRestore(str(folder))
    cb2.set_model(dst)
    st = fit_state(dst, 0)
    cb2.on_train_begin()
    assert st.epoch == 2 and st.history.history == {"loss": [0.5, 0.25]} and st.history.epoch == [0, 1]
    assert st.rng.get_state()[1].tolist() == st_src.rng.get_state()[1].tolist()
    assert _same(_snapshot(dst), _snapshot(src)) and dst.adam().iterations == 7
    # only the temporary file: nothing to restore
    os.remove(folder / BackupAndRestore.FILE)
    _, fresh = _models("BasicRS")
    fresh.compile()
    cb3 = BackupAndRestore(str(folder))
    cb3.set_model(fresh)
    st3 = fit_state(fresh, 0)
    cb3.on_train_begin()
    assert st3.epoch == 0 and fresh.count_params() == 0
    # another optimiser configuration: refused before the weights are written
    cb.on_epoch_end(1)
    other, _ = _models("BasicRS")
    other.compile(optimizer={"learning_rate": 1e-3})
    before = _snapshot(other)
    cb4 = BackupAndRestore(str(folder))
    cb4.set_model(other)
    fit_state(other, 0)
    with pytest.raises(ValueError, match="learning_rate"):
        cb4.on_train_begin()
    assert _same(_snapshot(other), before)
