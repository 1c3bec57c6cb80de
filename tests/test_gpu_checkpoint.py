"""Saving, loading and resuming on the GPU (keras_like.Model.save_weights / load_weights / fit(initial_epoch=) /
BackupAndRestore, training.Adam.state_dict / load_state_dict, the driver's model/weights.npz and
`backup_and_restore: true`).  Every training kernel is deterministic, so each comparison here is bit for bit.

1. Load = same model: a trained model saved and loaded into a fresh one built with another seed scores every pair, and
   ranks the whole catalog, with the same bits.
2. Resume = never stopped: fit(epochs=3) against fit(epochs=1) + save + load into a fresh model + fit(epochs=3,
   initial_epoch=1), and against a BackupAndRestore run whose process "dies" after epoch 0 (new model, new sequences):
   weights, Adam moments, iterations and the loss history, eager and with the CUDA-graphed step.
3. Partitioned: two processes on one GPU under a RowPartition resume bit-identically to the uninterrupted 2-rank and
   1-GPU runs; the 2-rank weight file loads into a 1-GPU model.
4. A captured GraphedTrainStep keeps working after load_weights / load_state_dict: its replay equals the eager step.
5. The driver: a run's model/weights.npz reproduces its test metrics; an interrupted backup_and_restore run started
   again ends with the metrics of an uninterrupted one."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NU, NI, NP = 61, 41, 17
CONTENT = 12
HYB_UNITS = [[16, 16], [16, 8], [16, 16]]
FAMILIES = ["BasicGCN", "BasicGAT", "BasicGraphSage", "BasicLightGCN", "BasicDGCF", "BasicRGCN",
            "HybridBertGCN-feature", "HybridBertGraphSage-entity", "BasicTSGCN", "BasicTWGCN", "BasicRS", "HybridCBRS"]
GNN_FAMILIES = [f for f in FAMILIES if f not in ("BasicRS", "HybridCBRS")]


@pytest.fixture(scope="module", autouse=True)
def _device():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)


class Data:
    """graphs, ratings and content rows shared by every model of a family"""

    def __init__(self, family):
        from deep_cbrs_amar_renaissance_b200.data.preprocess import get_user_properties
        from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
        from tests.helpers import kg_graphs
        self.family = family
        rng = np.random.RandomState(4)
        if family.startswith("BasicT"):
            self.nu, self.ni = 40, 30
            ui, ip = kg_graphs(self.nu, self.ni, 25)
            self.graph = (ui, ip, get_user_properties(ui, ip, self.nu, self.ni)) if "TW" in family else (ui, ip)
        else:
            self.nu, self.ni = NU, NI
            self.graph = small_graph(NU, NI, 700, seed=5, n_props=NP, n_links=120, dup_links=10)
            if family == "BasicRGCN":
                from tests.test_gpu_partitioned_training import _rgcn_graph
                self.graph = _rgcn_graph(self.graph, NU, NI, torch.device("cuda", 0))
        n = 900
        self.ratings = np.stack([rng.randint(0, self.nu, n), rng.randint(0, self.ni, n) + self.nu,
                                 rng.randint(0, 2, n)], axis=1).astype(np.int64)
        self.users, self.items = np.arange(self.nu), np.arange(self.ni)
        n_rows = self.nu + self.ni + NP
        self.content = (rng.standard_normal((n_rows, CONTENT)) * 0.5).astype(np.float32)
        self.graph_rows = (rng.standard_normal((n_rows, 10)) * 0.5).astype(np.float32)

    def model(self, seed, lr=1e-2):
        from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
        from deep_cbrs_amar_renaissance_b200.models import basic, hybrid
        set_seed(seed)
        f = self.family
        kw = dict(embedding_dim=8, n_hiddens=[8, 8], l2_regularizer=1e-4)
        if f.startswith("Hybrid") and f != "HybridCBRS":
            name, kind = f.split("-")
            m = getattr(hybrid, name)(self.graph, dense_units=HYB_UNITS, clf_units=[16, 16],
                                      feature_based=(kind == "feature"), **kw)
            m.set_content_table(self.content)
            m.build_weights(CONTENT)    # the graphed step of fit builds an unbuilt hybrid for 768-wide content
        elif f == "HybridCBRS":
            m = hybrid.HybridCBRS(feature_based=True, dense_units=HYB_UNITS, clf_units=[16, 16])
        elif f == "BasicRS":
            m = basic.BasicRS(dense_units=[16, 8], clf_units=[8])
        elif f.startswith("BasicT"):
            m = getattr(basic, f)(self.nu, self.ni, self.graph, dense_units=[16, 8], clf_units=[16, 16], **kw)
        elif f in ("BasicLightGCN", "BasicDGCF"):
            m = getattr(basic, f)(self.graph, n_layers=2, dense_units=[16, 8], clf_units=[16, 16], **kw)
        else:
            m = getattr(basic, f)(self.graph, dense_units=[16, 8], clf_units=[16, 16], **kw)
        m.compile(loss="binary_crossentropy", optimizer={"learning_rate": lr})
        return m

    def sequence(self):
        from deep_cbrs_amar_renaissance_b200.data import datasets as D
        args = (self.ratings, self.users, self.items)
        kw = dict(batch_size=128, shuffle=True, seed=9)
        if self.family == "BasicRS":
            return D.UserItemEmbeddings(*args, self.graph_rows, **kw)
        if self.family == "HybridCBRS":
            return D.HybridUserItemEmbeddings(*args, self.graph_rows, self.content, **kw)
        if self.family.startswith("Hybrid"):
            return D.UserItemGraphEmbeddings(*args, self.graph, self.content, device_resident=True, **kw)
        return D.UserItemGraph(*args, self.graph, **kw)

    def probe(self):
        """one batch of inputs to score"""
        u, i = self.ratings[:200, 0], self.ratings[:200, 1]
        if self.family == "BasicRS":
            return (self.graph_rows[u], self.graph_rows[i])
        if self.family == "HybridCBRS":
            return (self.graph_rows[u], self.graph_rows[i], self.content[u], self.content[i])
        return (u, i)


def _state(model):
    """(weights, Adam m, Adam v) by path, and iterations, on the host"""
    adam = model.adam().state_dict(model)
    torch.cuda.synchronize()
    host = lambda d: {k: v.detach().cpu().clone() for k, v in d.items()}  # noqa: E731
    return host(dict(model.named_weights())), host(adam["m"]), host(adam["v"]), adam["iterations"]


def _assert_same_state(got, want, what):
    for k, (a, b) in enumerate(zip(got[:3], want[:3])):
        assert list(a) == list(b), (what, ("weights", "m", "v")[k], sorted(set(a) ^ set(b)))
        for p in a:
            assert torch.equal(a[p], b[p]), "%s: %s %s differs" % (what, ("weight", "adam m", "adam v")[k], p)
    assert got[3] == want[3], (what, "iterations", got[3], want[3])


class _Die(Exception):
    pass


class DieAfterEpoch:
    """a callback that stops the process (here: fit) once epoch `epoch` has ended and been backed up"""

    def __init__(self, epoch):
        self.epoch = epoch

    def on_epoch_end(self, epoch, logs=None):
        if epoch == self.epoch:
            raise _Die()


# --------------------------------------------------------------------------------------------- 1. load = same model
@pytest.mark.parametrize("family", FAMILIES)
def test_a_loaded_model_scores_and_ranks_with_the_same_bits(tmp_path, family):
    d = Data(family)
    m = d.model(1)
    m.fit(d.sequence(), epochs=1)
    path = str(tmp_path / "weights.npz")
    m.save_weights(path)
    fresh = d.model(2)
    fresh.load_weights(path)
    x = d.probe()
    assert torch.equal(fresh(x), m(x))
    if family in GNN_FAMILIES:
        users = torch.arange(d.nu, device="cuda")
        a_ids, a_val = m.recommend_top_k(d.nu, d.ni, 10, users=users)
        b_ids, b_val = fresh.recommend_top_k(d.nu, d.ni, 10, users=users)
        assert torch.equal(a_ids, b_ids) and torch.equal(a_val, b_val)


# ------------------------------------------------------------------------------------------ 2. resume = never stopped
@pytest.mark.parametrize("cuda_graph", [False, True], ids=["eager", "graphed"])
@pytest.mark.parametrize("family", FAMILIES)
def test_a_resumed_fit_equals_the_fit_that_never_stopped(tmp_path, family, cuda_graph):
    d = Data(family)
    ref = d.model(1)
    want_hist = ref.fit(d.sequence(), epochs=3, cuda_graph=cuda_graph).history["loss"]
    want = _state(ref)
    assert len(want_hist) == 3 and want[3] == 3 * len(d.sequence())

    # save after epoch 0, load into a fresh model, continue with initial_epoch=1 (same sequence object)
    first, seq = d.model(1), d.sequence()
    h0 = first.fit(seq, epochs=1, cuda_graph=cuda_graph).history["loss"]
    first.save_weights(str(tmp_path / "weights.npz"))
    adam = first.adam().state_dict(first)
    adam = dict(adam, m={k: v.cpu().numpy() for k, v in adam["m"].items()},
                v={k: v.cpu().numpy() for k, v in adam["v"].items()})
    second = d.model(2)
    second.load_weights(str(tmp_path / "weights.npz"))
    second.adam().load_state_dict(second, adam)
    h12 = second.fit(seq, epochs=3, initial_epoch=1, cuda_graph=cuda_graph).history["loss"]
    assert h0 + h12 == want_hist
    _assert_same_state(_state(second), want, "initial_epoch")

    # BackupAndRestore: the process dies after epoch 0; a new one (new model, new sequence) starts the same fit
    from deep_cbrs_amar_renaissance_b200.keras_like import BackupAndRestore
    backup = str(tmp_path / "backup")
    with pytest.raises(_Die):
        d.model(1).fit(d.sequence(), epochs=3, cuda_graph=cuda_graph,
                       callbacks=[BackupAndRestore(backup), DieAfterEpoch(0)])
    assert os.listdir(backup) == [BackupAndRestore.FILE]
    resumed = d.model(2)
    hist = resumed.fit(d.sequence(), epochs=3, cuda_graph=cuda_graph, callbacks=[BackupAndRestore(backup)])
    assert hist.history["loss"] == want_hist and hist.epoch == [0, 1, 2]
    _assert_same_state(_state(resumed), want, "BackupAndRestore")
    assert os.listdir(backup) == []            # deleted when training ends


# ------------------------------------------------------------------------------------------------- 3. partitioned
PART_FAMILIES = ["BasicGCN", "HybridBertGCN-feature"]


def _part_worker(rank, world, init, out_dir):
    import torch.distributed as dist
    from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
    from deep_cbrs_amar_renaissance_b200.keras_like import BackupAndRestore
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    failures, cases = [], 0

    def check(what, fn):
        nonlocal cases
        cases += 1
        try:
            fn()
        except AssertionError as e:
            failures.append("%s: %s" % (what, e))

    try:
        for family in PART_FAMILIES:
            d = Data(family)
            sizes = (NU, NI, NP)

            def partitioned(seed):
                m = d.model(seed)
                RowPartition(sizes, exchange="nccl").attach(m.gnn.gnn_layers)
                return m

            one = d.model(1)
            h1 = one.fit(d.sequence(), epochs=3).history["loss"]
            want = _state(one)
            full = partitioned(1)
            h2 = full.fit(d.sequence(), epochs=3).history["loss"]
            backup = os.path.join(out_dir, family, "backup")
            try:
                partitioned(1).fit(d.sequence(), epochs=3, callbacks=[BackupAndRestore(backup), DieAfterEpoch(0)])
            except _Die:
                pass
            resumed = partitioned(2)
            h3 = resumed.fit(d.sequence(), epochs=3, callbacks=[BackupAndRestore(backup)]).history["loss"]
            check(family + " 2-rank run vs 1 GPU", lambda: (_assert_same_state(_state(full), want, "2 ranks"),
                                                           (h2 == h1) or _fail("loss history %s vs %s" % (h2, h1))))
            check(family + " resumed 2-rank run vs 1 GPU", lambda: (_assert_same_state(_state(resumed), want, "resumed"),
                                                                   (h3 == h1) or _fail("loss history %s vs %s" % (h3, h1))))
            path = os.path.join(out_dir, family, "weights.npz")
            if rank == 0:
                resumed.save_weights(path)
            dist.barrier()
            single = d.model(3)
            single.load_weights(path)
            check(family + " 2-rank file into a 1-GPU model", lambda: _assert_same_state(
                (dict((k, v.cpu()) for k, v in single.named_weights()), {}, {}, 0), (want[0], {}, {}, 0), "loaded"))
            dist.barrier()
    finally:
        with open(os.path.join(out_dir, "rank%d.json" % rank), "w") as f:
            json.dump({"cases": cases, "failures": failures}, f)
        dist.destroy_process_group()


def _fail(msg):
    raise AssertionError(msg)


def test_partitioned_runs_resume_bit_identically(tmp_path):
    """two processes share cuda:0 and a gloo group (as in test_gpu_partitioned_training.py): rank 0 writes the backup,
    both ranks restore it"""
    import torch.multiprocessing as mp
    mp.spawn(_part_worker, args=(2, "file://" + str(tmp_path / "store"), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        res = json.load(open(tmp_path / ("rank%d.json" % r)))
        assert res["cases"] == 3 * len(PART_FAMILIES) and not res["failures"], res["failures"]


# ------------------------------------------------------------------------------------------- 4. graph slots survive
@pytest.mark.parametrize("family", ["BasicGCN", "HybridBertGCN-feature"])
def test_a_captured_step_reads_the_loaded_weights_and_moments(tmp_path, family):
    d = Data(family)
    seq = d.sequence()
    src = d.model(1)
    src.fit(seq, epochs=1)
    path = str(tmp_path / "weights.npz")
    src.save_weights(path)
    adam = src.adam().state_dict(src)
    (u, i), y = seq[0]

    graphed = d.model(2)
    graphed.build_weights(CONTENT) if family.startswith("Hybrid") else graphed.build_weights()
    step = graphed.make_graphed_train_step(len(y))
    slots = {id(w): graphed.adam()._state[id(w)] for w in graphed.weights if id(w) in graphed.adam()._state}
    weights = [w.data_ptr() for w in graphed.weights]
    graphed.load_weights(path)
    graphed.adam().load_state_dict(graphed, adam)
    assert [w.data_ptr() for w in graphed.weights] == weights
    assert all(graphed.adam()._state[k] is s for k, s in slots.items())

    eager = d.model(3)
    eager.load_weights(path)
    eager.adam().load_state_dict(eager, adam)
    for k in range(2):
        (u, i), y = seq[k]
        lg, _ = step((u, i), y)
        le, _ = eager.train_on_batch((u, i), y)
        assert torch.equal(lg, le)
    _assert_same_state(_state(graphed), _state(eager), "graphed after load")


# ----------------------------------------------------------------------------------------------------- 5. driver
COMPARED = ("test_loss", "test_accuracy", "history") + tuple("%s_at_%d" % (m, k) for m in ("precision", "recall", "f1")
                                                             for k in (5, 10))


def _driver_inputs(root, backup):
    import yaml
    from tests.test_zz_gpu_experiment import write_inputs
    cfg, _, paths = write_inputs(root)
    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    base = ex.load_yaml(cfg)
    base["catalog_metrics"] = True
    if backup:
        base["backup_and_restore"] = True
    base["model"]["name"] = "basic.BasicGCN"
    base["dataset"]["load_function_name"] = "load_user_item_graph"
    with open(cfg, "w") as fp:
        yaml.safe_dump(base, fp)
    exps = os.path.join(str(root), "one.yaml")
    with open(exps, "w") as fp:
        yaml.safe_dump({"linear": {"gcn": None}}, fp)
    return cfg, exps


def _catalog_keys(m):
    return [k for k in m if k.startswith("catalog_")]


def test_driver_writes_weights_that_reproduce_the_run(tmp_path):
    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    cfg, exps = _driver_inputs(tmp_path / "data", backup=False)
    res = ex.main(["-c", cfg, "-e", exps, "--out", str(tmp_path / "runs"), "--exp_name", "w"])["gcn"]
    assert res is not None and _catalog_keys(res)
    (run,) = os.listdir(tmp_path / "runs" / "w")
    run_dir = tmp_path / "runs" / "w" / run
    weights = run_dir / "model" / ex.WEIGHTS_FILE
    assert weights.exists()
    config = ex.load_yaml(str(run_dir / "artifacts" / "config.yaml"))
    again = ex.Experimenter(config, str(tmp_path / "reload"))
    again.build_dataset()
    again.build_optimizer()
    again.build_model()
    again.model.load_weights(str(weights))
    again.evaluate()
    again.close()
    for k in ("test_loss", "test_accuracy") + COMPARED[3:] + tuple(_catalog_keys(res)):
        assert again.metrics[k] == res[k], k


def test_driver_resumes_an_interrupted_run(tmp_path, monkeypatch):
    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    from deep_cbrs_amar_renaissance_b200.keras_like import BackupAndRestore
    cfg, exps = _driver_inputs(tmp_path / "data", backup=True)
    want = ex.main(["-c", cfg, "-e", exps, "--out", str(tmp_path / "a"), "--exp_name", "r"])["gcn"]
    assert want is not None and len(want["history"]["loss"]) == 3
    args = ["-c", cfg, "-e", exps, "--out", str(tmp_path / "b"), "--exp_name", "r"]
    original = BackupAndRestore.on_epoch_end

    def dies_after_epoch_0(self, epoch, logs=None):
        original(self, epoch, logs)
        if epoch == 0:
            raise _Die()

    monkeypatch.setattr(BackupAndRestore, "on_epoch_end", dies_after_epoch_0)
    assert ex.main(args)["gcn"] is None
    (run,) = os.listdir(tmp_path / "b" / "r")
    assert os.listdir(tmp_path / "b" / "r" / run / "backup") == [BackupAndRestore.FILE]
    monkeypatch.setattr(BackupAndRestore, "on_epoch_end", original)
    got = ex.main(args)["gcn"]
    assert os.listdir(tmp_path / "b" / "r") == [run]            # the same run, continued in its directory
    saved = json.load(open(tmp_path / "b" / "r" / run / "artifacts" / "metrics.json"))
    for k in COMPARED + tuple(_catalog_keys(want)):
        assert got[k] == want[k] and saved[k] == want[k], k
