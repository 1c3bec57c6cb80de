"""Save / load time and file size of a model's weights and of its whole training state at config-5 size.

BasicGCN, embedding width 128 and three 128-wide GCN layers, over a 1.1e7-node graph (the table is 1.1e7 x 128 fp32,
5.6 GB; with the two Adam moments the training state is about 17 GB).  One optimiser step creates the moments; the
graph has few edges, since only the sizes of the saved arrays matter here.  Measured:
  * Model.save_weights / Model.load_weights (into a fresh model) of the weights alone;
  * BackupAndRestore's epoch-end write and train-begin restore of the training state (weights + Adam moments).
Each time ends in a device synchronise; each load is checked bit for bit.  Files go to a temporary directory (or
--dir) and are deleted afterwards.

    python tools/checkpoint_bench.py [--nodes 11000000] [--dir /path] [--out result.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=11_000_000)
    ap.add_argument("--width", type=int, default=128)
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from scipy import sparse

    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.keras_like import BackupAndRestore, History, _FitState, set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic
    ops.check_device()
    torch.cuda.set_device(0)
    n, w = args.nodes, args.width
    n_users = n // 2
    rng = np.random.RandomState(0)
    r = rng.randint(0, n_users, n).astype(np.int32)
    c = (rng.randint(0, n - n_users, n) + n_users).astype(np.int32)
    adj = sparse.coo_matrix((np.ones(2 * n, np.float32), (np.concatenate([r, c]), np.concatenate([c, r]))),
                            shape=(n, n))

    def model(seed):
        set_seed(seed)
        m = basic.BasicGCN(adj, embedding_dim=w, n_hiddens=[w, w, w], dense_units=[64, 64], clf_units=[64, 64])
        m.compile(optimizer={"learning_rate": 1e-3})
        return m

    src = model(1)
    src.build_weights()
    u = rng.randint(0, n_users, 4096)
    i = rng.randint(n_users, n, 4096)
    src.train_on_batch((u, i), (rng.rand(4096) < 0.5).astype(np.float32))
    torch.cuda.synchronize()
    folder = tempfile.mkdtemp(prefix="cbrs_ckpt_", dir=args.dir)
    res = dict(card(), nodes=n, width=w, params=src.count_params())
    try:
        def timed(fn):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            return time.perf_counter() - t

        path = os.path.join(folder, "weights.npz")
        res["weights_save_s"] = timed(lambda: src.save_weights(path))
        res["weights_file_bytes"] = os.path.getsize(path)
        dst = model(2)
        res["weights_load_s"] = timed(lambda: dst.load_weights(path))
        res["weights_bit_identical"] = all(torch.equal(a, b) for a, b in zip(src.weights, dst.weights))
        del dst
        os.remove(path)
        torch.cuda.empty_cache()

        def fit_state(m):
            m._fit_state = _FitState(None, np.random.RandomState(m.shuffle_seed), History(), 0)

        cb = BackupAndRestore(os.path.join(folder, "backup"))
        cb.set_model(src)
        fit_state(src)
        res["state_save_s"] = timed(lambda: cb.on_epoch_end(0))
        res["state_file_bytes"] = os.path.getsize(cb.path)
        dst = model(3)
        fit_state(dst)
        cb2 = BackupAndRestore(os.path.join(folder, "backup"))
        cb2.set_model(dst)
        res["state_load_s"] = timed(cb2.on_train_begin)
        sa, sb = src.adam().state_dict(src), dst.adam().state_dict(dst)
        res["state_bit_identical"] = (all(torch.equal(a, b) for a, b in zip(src.weights, dst.weights))
                                      and all(torch.equal(sa[k][p], sb[k][p]) for k in "mv" for p in sa[k])
                                      and sa["iterations"] == sb["iterations"] and sorted(sa["m"]) == sorted(sb["m"]))
    finally:
        shutil.rmtree(folder, ignore_errors=True)
    for k in ("weights", "state"):
        res[k + "_save_GBps"] = res[k + "_file_bytes"] / res[k + "_save_s"] / 1e9
        res[k + "_load_GBps"] = res[k + "_file_bytes"] / res[k + "_load_s"] / 1e9
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
