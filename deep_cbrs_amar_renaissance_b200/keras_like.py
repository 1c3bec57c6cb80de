"""The slice of the Keras Layer/Model surface the reference's caller uses
(/root/reference/src/experiment.py:136-197, src/utilities/keras.py:10-22):
add_weight, lazy build, trainable_weights, get/set_weights, compile, __call__,
summary, evaluate, predict.  Weights are float32 CUDA tensors; initialisers follow
Keras (glorot_uniform / zeros / ones) and are drawn on the host from one seeded
generator so a run is reproducible across devices.
"""
import math
import os
from collections import OrderedDict

import numpy as np
import torch

_GEN = torch.Generator(device="cpu")
_GEN.manual_seed(42)


def set_seed(seed):
    """Counterpart of tf.random.set_seed (experiment.py:56)."""
    _GEN.manual_seed(int(seed))


def default_device():
    """CUDA device of this process.  Without CUDA, weights can still be CREATED on the host
    (shape / parameter-count logic); every op refuses non-CUDA tensors, so nothing computes."""
    if not torch.cuda.is_available():
        return torch.device("cpu")
    return torch.device("cuda", torch.cuda.current_device())


def _init(shape, initializer):
    shape = tuple(int(s) for s in shape)
    if initializer == "zeros":
        return torch.zeros(shape, dtype=torch.float32)
    if initializer == "ones":
        return torch.ones(shape, dtype=torch.float32)
    if initializer == "glorot_uniform":
        # Keras: fan_in = shape[-2] * receptive field, fan_out = shape[-1] * receptive field
        if len(shape) == 1:
            fan_in = fan_out = shape[0]
        else:
            rf = int(np.prod(shape[:-2])) if len(shape) > 2 else 1
            fan_in, fan_out = shape[-2] * rf, shape[-1] * rf
        limit = math.sqrt(6.0 / (fan_in + fan_out))
        return (torch.rand(shape, generator=_GEN, dtype=torch.float32) * 2.0 - 1.0) * limit
    raise ValueError("initializer not supported: {}".format(initializer))


class L2:
    """regularizers.l2(l): penalty l * sum(w^2) (src/models/gnn.py:239-246)."""

    def __init__(self, l2):
        self.l2 = float(l2)


class Layer:
    def __init__(self, name=None):
        self.name = name or type(self).__name__.lower()
        self._weights = OrderedDict()
        self._regularizers = {}
        self.built = False

    # -- weights ---------------------------------------------------------
    def add_weight(self, name, shape, initializer="glorot_uniform", regularizer=None, trainable=True):
        dev = default_device()
        if initializer == "glorot_uniform" and int(np.prod(shape)) > (1 << 24) and dev.type == "cuda":
            # large tables (scaled graphs): draw on the device from a generator seeded by the host one
            gen = torch.Generator(device=dev)
            gen.manual_seed(int(torch.randint(0, 2 ** 31 - 1, (1,), generator=_GEN).item()))
            limit = math.sqrt(6.0 / (int(shape[-2]) + int(shape[-1])))
            w = torch.rand(tuple(int(v) for v in shape), generator=gen, dtype=torch.float32, device=dev)
            w.mul_(2.0 * limit).sub_(limit)
        else:
            w = _init(shape, initializer).to(dev)
        w.trainable = trainable
        self._weights[name] = w
        if regularizer is not None:
            self._regularizers[name] = regularizer
        return w

    def _sublayers(self):
        """(attribute path, layer) of every directly owned sub-layer, in attribute order."""
        out, seen = [], []
        for attr, v in self.__dict__.items():
            items = [(attr, v)] if not isinstance(v, (list, tuple)) else [("%s.%d" % (attr, k), it) for k, it in enumerate(v)]
            for path, it in items:
                if isinstance(it, Layer) and it is not self and all(it is not s for s in seen):
                    seen.append(it)
                    out.append((path, it))
        return out

    def named_weights(self, prefix=""):
        """[(path, tensor)]: own weights first, then sub-layers by attribute path,
        e.g. 'gnn/gnn_layers/seq_layers.0/kernel', 'rs/unet/layers.1/bias'."""
        out = [(prefix + k, v) for k, v in self._weights.items()]
        for path, sub in self._sublayers():
            out.extend(sub.named_weights(prefix + path + "/"))
        return out

    @property
    def weights(self):
        return [w for _, w in self.named_weights()]

    @property
    def trainable_weights(self):
        return [w for w in self.weights if getattr(w, "trainable", True)]

    @property
    def non_trainable_weights(self):
        return [w for w in self.weights if not getattr(w, "trainable", True)]

    def get_weights(self):
        return [w.detach().cpu().numpy() for w in self.weights]

    def set_weights(self, arrays):
        ws = self.weights
        if len(ws) != len(arrays):
            raise ValueError("expected {} arrays, got {}".format(len(ws), len(arrays)))
        for w, a in zip(ws, arrays):
            a = torch.as_tensor(np.asarray(a, dtype=np.float32))
            if tuple(a.shape) != tuple(w.shape):
                raise ValueError("shape mismatch {} vs {}".format(tuple(a.shape), tuple(w.shape)))
            w.copy_(a.to(w.device))

    def count_params(self):
        return int(sum(w.numel() for w in self.weights))

    # -- call ------------------------------------------------------------
    def build(self, input_shape):
        self.built = True

    def call(self, inputs, **kwargs):
        raise NotImplementedError

    def __call__(self, inputs, **kwargs):
        if not self.built:
            self.build(_shape_of(inputs))
            self.built = True
        return self.call(inputs, **kwargs)


def _shape_of(x):
    if isinstance(x, (list, tuple)):
        return [_shape_of(v) for v in x]
    return tuple(x.shape) if hasattr(x, "shape") else None


class History:
    """What keras `fit` returns: `.history[name]` = one value per epoch."""

    def __init__(self):
        self.history = {}
        self.epoch = []


class _FitState:
    """The loop state of a running `fit`: the sequence, the batch-order RandomState, the History and the next epoch."""

    def __init__(self, sequence, rng, history, epoch):
        self.sequence, self.rng, self.history, self.epoch = sequence, rng, history, epoch


def _row_partition(model):
    """The RowPartition attached to one of the model's GNN stacks, or None."""
    from .models.gnn import SequentialGNN
    gnn = getattr(model, "gnn", None)
    for s in (vars(gnn).values() if gnn is not None else ()):
        if isinstance(s, SequentialGNN) and s.partition is not None:
            return s.partition
    return None


class BackupAndRestore:
    """keras.callbacks.BackupAndRestore(backup_dir): lets a training run that stopped continue where it stopped.

    At every epoch end the training state goes to <backup_dir>/training_state.npz, written under a temporary name
    and renamed over the previous one (checkpoint.write), so a run killed mid-write leaves the previous epoch's file.
    At train begin a state found there is restored and `fit` continues with the epoch after the saved one.  The
    state: the weights, the Adam moments and iteration count, the epoch index, fit's batch-order RandomState, the
    sequence's RandomState(s) and row order, and the History so far.  Every kernel of a step is deterministic, so the
    resumed run computes the bits of the run that never stopped.  The file is deleted when training ends.

    Under a RowPartition every rank holds the same weights and moments bit for bit: rank 0 writes, then the ranks
    meet at a barrier, and every rank restores from the same file."""

    FILE = "training_state.npz"

    def __init__(self, backup_dir):
        self.backup_dir = backup_dir
        self.path = os.path.join(backup_dir, self.FILE)
        self.model = None

    def set_model(self, model):
        self.model = model

    def _rank_and_group(self):
        part = _row_partition(self.model)
        return (0, None) if part is None else (part.rank, part)

    def _barrier(self, part):
        if part is not None:
            import torch.distributed as dist
            dist.barrier(group=part.group)

    def _sequence_state(self, st):
        get = getattr(st.sequence, "get_state", None)
        return get() if get is not None else {}

    def on_train_begin(self, logs=None):
        from . import checkpoint
        if not os.path.exists(self.path):
            return
        m, st = self.model, self.model._fit_state
        adam = m.adam()
        with checkpoint.Reader(self.path, "training_state") as rd:
            h = rd.header
            m._check_weight_arrays(rd, rd.arrays("weights/"))
            seq = rd.arrays("sequence/")
            checkpoint.check_arrays(self.path + " (sequence state)",
                                    checkpoint.spec(self._sequence_state(st).items()), seq)
            checkpoint.check_arrays(self.path + " (fit batch order)",
                                    checkpoint.spec(checkpoint.rng_arrays(st.rng).items()), rd.arrays("fit/"))
            # checks the Adam hyper-parameters and moments before writing anything, so nothing is written on a refusal
            adam.load_state_dict(m, dict(h["adam"], m=rd.arrays("adam/m/"), v=rd.arrays("adam/v/")))
            m._copy_weights(rd.arrays("weights/"))
            if seq:
                st.sequence.set_state(seq)
            checkpoint.set_rng(st.rng, rd.arrays("fit/"))
            st.history.history = {k: list(v) for k, v in h["history"].items()}
            st.history.epoch = list(h["history_epochs"])
            st.epoch = int(h["epoch"]) + 1

    def on_epoch_end(self, epoch, logs=None):
        from . import checkpoint
        rank, part = self._rank_and_group()
        if rank == 0:
            m, st = self.model, self.model._fit_state
            adam = m.adam().state_dict(m)
            arrays = [("weights/" + p, w) for p, w in m.named_weights()]
            arrays += [("adam/m/" + p, t) for p, t in adam.pop("m").items()]
            arrays += [("adam/v/" + p, t) for p, t in adam.pop("v").items()]
            arrays += [("sequence/" + k, a) for k, a in self._sequence_state(st).items()]
            arrays += [("fit/" + k, a) for k, a in checkpoint.rng_arrays(st.rng).items()]
            header = {"kind": "training_state", "version": checkpoint.VERSION, "model": type(m).__name__,
                      "epoch": int(epoch), "adam": adam, "history": st.history.history,
                      "history_epochs": st.history.epoch}
            checkpoint.write(self.path, header, arrays)
        self._barrier(part)

    def on_train_end(self, logs=None):
        rank, part = self._rank_and_group()
        self._barrier(part)
        if rank == 0 and os.path.exists(self.path):
            os.remove(self.path)


class Model(Layer):
    """compile / fit / predict / evaluate / summary as the reference's Experimenter calls them
    (/root/reference/src/experiment.py:155-197)."""

    loss = optimizer = metrics = None
    shuffle_seed = 42  # Keras shuffles the batch order of a Sequence with an unseeded RNG; ours is seeded

    def compile(self, loss=None, optimizer=None, metrics=None):
        if loss not in (None, "binary_crossentropy", "BinaryCrossentropy"):
            raise NotImplementedError("loss '{}': the reference trains with binary_crossentropy "
                                      "(config.yaml:50)".format(loss))
        self.loss, self.optimizer, self.metrics = loss, optimizer, metrics
        self._adam = None

    def adam(self):
        """The optimiser the training steps update (created from the compiled config at first use)."""
        from . import training
        if getattr(self, "_adam", None) is None:
            self._adam = training.Adam.from_config(self.optimizer)
        return self._adam

    def train_on_batch(self, x, y):
        """One optimiser step; returns (loss incl. l2 penalty, #correct) as device scalars."""
        from . import training
        return training.train_step(self, self.adam(), x, y)

    def make_graphed_train_step(self, batch_size, content_dim=None):
        """CUDA-graph replay of the whole optimiser step for a fixed batch size (training.GraphedTrainStep)."""
        from . import training
        return training.GraphedTrainStep(self, self.adam(), batch_size, content_dim)

    # -- weight files ----------------------------------------------------
    def build_from_shapes(self, shapes):
        """Create the weights for a file whose arrays have `shapes` ({weight path: shape}).  The GNN models build
        from their constructor arguments; the scorers and hybrids override this to read their input widths."""
        self.build_weights()

    def save_weights(self, path):
        """Write every weight to `path` (a .npz, see checkpoint.py), keyed by its path in named_weights(), with a
        header naming the model class and each path's shape and dtype.  Not saved, because they are data or settings
        rather than weights: the content table (set_content_table), the scorer precision and the feature dtype."""
        from . import checkpoint
        named = self.named_weights()
        checkpoint.write(path, {"kind": "weights", "version": checkpoint.VERSION, "model": type(self).__name__,
                                "weights": checkpoint.spec(named)}, named)

    def load_weights(self, path):
        """Read a file of save_weights into this model, building its weights first if needed.  Refuses, before any
        weight is written, a file of another model class, and a missing path, an extra path or a shape or dtype
        mismatch, naming the first offending path.  Copies in place: tensors captured by a GraphedTrainStep stay
        valid."""
        from . import checkpoint
        with checkpoint.Reader(path, "weights") as rd:
            self._check_weight_arrays(rd, rd.arrays())
            self._copy_weights(rd.arrays())

    def _check_weight_arrays(self, reader, arrays):
        from . import checkpoint
        if reader.header["model"] != type(self).__name__:
            raise ValueError("{}: written by a {}, this model is a {}".format(reader.path, reader.header["model"],
                                                                             type(self).__name__))
        self.build_from_shapes({k: tuple(a.shape) for k, a in arrays.items()})
        checkpoint.check_arrays(reader.path, checkpoint.spec(self.named_weights()), arrays)

    def _copy_weights(self, arrays):
        for name, w in self.named_weights():
            w.copy_(torch.from_numpy(np.asarray(arrays[name])))
        if hasattr(self, "invalidate"):
            self.invalidate()

    def predict(self, sequence):
        outs = []
        for i in range(len(sequence)):
            x, _ = sequence[i]
            outs.append(self(x).detach().cpu().numpy())
        return np.concatenate(outs, axis=0)

    def evaluate(self, sequence):
        """[binary cross-entropy, accuracy] averaged over samples (Keras clips p to [1e-7, 1-1e-7])."""
        loss = acc = n = 0.0
        for i in range(len(sequence)):
            x, y = sequence[i]
            p = self(x).detach().cpu().numpy().reshape(-1).astype(np.float64)
            y = np.asarray(y, dtype=np.float64).reshape(-1)
            pc = np.clip(p, 1e-7, 1 - 1e-7)
            loss += float(-(y * np.log(pc) + (1 - y) * np.log(1 - pc)).sum())
            acc += float(((p > 0.5) == (y > 0.5)).sum())
            n += len(y)
        return [loss / max(n, 1), acc / max(n, 1)]

    def fit(self, sequence, epochs=1, workers=1, callbacks=None, shuffle=True, verbose=0, cuda_graph=False,
            initial_epoch=0):
        """Keras `fit` over a `Sequence` (/root/reference/src/experiment.py:183-188): per epoch every batch
        once, in shuffled batch order, `sequence.on_epoch_end()` after the last one (the reference's
        datasets reshuffle their rows there, src/data/datasets.py:205-213); callbacks receive the Keras
        hooks the reference's own callbacks implement (src/utilities/keras.py:43-90).  `workers` is accepted
        and ignored (batches are index slices of an in-memory array).  cuda_graph=True replays full-size
        batches through one captured CUDA graph of the whole step (same kernels, same results); a short last
        batch runs eagerly.

        initial_epoch: the epoch to start at (Keras): epochs initial_epoch .. epochs-1 run.  The batch order of an
        epoch depends only on its index, so a model and sequences saved after epoch k-1 and trained on with
        initial_epoch=k replay the batches of the run that never stopped.  A BackupAndRestore callback that finds a
        saved state sets the start epoch itself."""
        from . import training
        training.check_not_partitioned_build(self)
        callbacks = list(callbacks or [])
        hist = History()
        rng = np.random.RandomState(self.shuffle_seed)
        if shuffle:
            for _ in range(int(initial_epoch)):
                rng.permutation(len(sequence))
        # what a BackupAndRestore callback saves and restores besides the weights and the optimiser
        self._fit_state = _FitState(sequence, rng, hist, int(initial_epoch))

        def fire(name, *args):
            for cb in callbacks:
                fn = getattr(cb, name, None)
                if fn is not None:
                    fn(*args)

        for cb in callbacks:
            if hasattr(cb, "set_model"):
                cb.set_model(self)
            else:
                cb.model = self
        graphed = None
        fire("on_train_begin", {})
        logs = {}
        for epoch in range(self._fit_state.epoch, int(epochs)):
            fire("on_epoch_begin", epoch, {})
            order = rng.permutation(len(sequence)) if shuffle else np.arange(len(sequence))
            losses, corrects, sizes = [], [], []
            for step, b in enumerate(order):
                x, y = sequence[int(b)]
                fire("on_train_batch_begin", step, {})
                if cuda_graph and len(x) == 2 and hasattr(self, 'gnn'):
                    if graphed is None and len(sequence) > 1:
                        graphed = self.make_graphed_train_step(len(sequence[0][1]))
                    if graphed is not None and len(y) == graphed.batch_size:
                        loss, correct = graphed(x, y)
                    else:
                        loss, correct = self.train_on_batch(x, y)
                else:
                    loss, correct = self.train_on_batch(x, y)
                losses.append(loss)
                corrects.append(correct)
                sizes.append(len(y))
                fire("on_train_batch_end", step, {})
            n = float(sum(sizes))
            lv = torch.cat(losses).double().cpu().numpy()
            cv = torch.cat(corrects).double().cpu().numpy()
            logs = {"loss": float((lv * np.asarray(sizes)).sum() / n), "accuracy": float(cv.sum() / n)}
            for k, v in logs.items():
                hist.history.setdefault(k, []).append(v)
            hist.epoch.append(epoch)
            if hasattr(sequence, "on_epoch_end"):
                sequence.on_epoch_end()
            if verbose:
                print("epoch {}: {}".format(epoch + 1, logs))
            self._fit_state.epoch = epoch + 1
            fire("on_epoch_end", epoch, logs)
        fire("on_train_end", logs)
        self._fit_state = None
        return hist

    def summary(self, print_fn=print, expand_nested=True):
        print_fn("Model: {}".format(type(self).__name__))
        for name, w in self.named_weights():
            print_fn("  {:60s} {:>18s} {:>10d}".format(name, str(tuple(w.shape)), w.numel()))
        print_fn("Total params: {}".format(self.count_params()))
