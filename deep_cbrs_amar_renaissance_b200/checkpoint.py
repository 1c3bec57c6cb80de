"""The file format of saved weights and training states.

A checkpoint is a numpy .npz archive (a zip of .npy members, stored uncompressed) that `np.load(path,
allow_pickle=False)` reads: loading it executes no code.  The member "header" holds the JSON header as uint8 bytes;
every other member is one array keyed by its path, e.g. "gnn/gnn_layers/seq_layers.0/kernel".  float32 arrays are
stored exactly as the device holds them.

Arrays are copied from the device and written one at a time, and read back one at a time, so the host holds one array
of a model rather than all of them (a config-5 embedding table alone is 5.6 GB).  A file is written under a temporary
name in the target directory, flushed to disk and renamed over the target: a reader finds the previous file or the
new one, never a partly written one."""
import json
import os
import tempfile
import zipfile

import numpy as np

VERSION = 1
HEADER = "header"


def _host(a):
    if isinstance(a, np.ndarray):
        return np.ascontiguousarray(a)
    return a.detach().contiguous().cpu().numpy()


def write(path, header, arrays):
    """header: a JSON-serialisable dict; arrays: iterable of (name, torch tensor or ndarray)."""
    path = os.path.abspath(path)
    folder = os.path.dirname(path)
    os.makedirs(folder, exist_ok=True)
    fd, tmp = tempfile.mkstemp(prefix="." + os.path.basename(path) + ".", suffix=".tmp", dir=folder)
    try:
        with os.fdopen(fd, "wb") as fp:
            with zipfile.ZipFile(fp, "w", zipfile.ZIP_STORED, allowZip64=True) as zf:
                names = set()
                for name, a in [(HEADER, np.frombuffer(json.dumps(header).encode(), np.uint8))] + list(arrays):
                    if name in names:
                        raise ValueError("two arrays named '{}'".format(name))
                    names.add(name)
                    with zf.open(name + ".npy", "w", force_zip64=True) as f:
                        np.lib.format.write_array(f, _host(a), allow_pickle=False)
            fp.flush()
            os.fsync(fp.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise


class StoredArray:
    """One member of an open checkpoint: shape and dtype from its .npy header; the data is read by np.asarray."""

    def __init__(self, npz, name, shape, dtype):
        self._npz, self.name, self.shape, self.dtype = npz, name, tuple(shape), np.dtype(dtype)

    def __array__(self, dtype=None, copy=None):
        a = self._npz[self.name]
        return a if dtype is None else a.astype(dtype)


def _npy_meta(zf, member):
    with zf.open(member) as f:
        version = np.lib.format.read_magic(f)
        readers = {(1, 0): np.lib.format.read_array_header_1_0, (2, 0): np.lib.format.read_array_header_2_0}
        if version not in readers:
            raise ValueError("member '{}': .npy format version {} is not supported".format(member, version))
        shape, _, dtype = readers[version](f)
    return shape, dtype


class Reader:
    """An open checkpoint: `header`, and `arrays(prefix)` -> {name without the prefix: StoredArray}.  Opening reads
    the header and every member's .npy header, no array data."""

    def __init__(self, path, kind):
        self.path = path
        self._npz = np.load(path, allow_pickle=False)
        try:
            if HEADER not in self._npz.files:
                raise ValueError("{}: not a checkpoint (no '{}' member)".format(path, HEADER))
            self.header = json.loads(np.asarray(self._npz[HEADER]).tobytes().decode())
            if self.header.get("kind") != kind:
                raise ValueError("{}: holds '{}', expected '{}'".format(path, self.header.get("kind"), kind))
            if self.header.get("version") != VERSION:
                raise ValueError("{}: format version {}, this library reads {}".format(
                    path, self.header.get("version"), VERSION))
            self._members = {}
            for name in self._npz.files:
                if name != HEADER:
                    shape, dtype = _npy_meta(self._npz.zip, name + ".npy")
                    self._members[name] = StoredArray(self._npz, name, shape, dtype)
        except BaseException:
            self._npz.close()
            raise

    def arrays(self, prefix=""):
        return {k[len(prefix):]: v for k, v in self._members.items() if k.startswith(prefix)}

    def close(self):
        self._npz.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def dtype_name(a):
    """'float32' for a float32 ndarray, torch tensor or StoredArray"""
    return str(a.dtype).replace("torch.", "")


def check_arrays(what, want, got):
    """want: [(name, shape, dtype name)] in order; got: {name: array-like with .shape and .dtype}.  Raises ValueError
    naming the first name that is missing, has another shape or dtype, or (after every wanted name) is extra."""
    names = set()
    for name, shape, dtype in want:
        names.add(name)
        if name not in got:
            raise ValueError("{}: '{}' is missing".format(what, name))
        a = got[name]
        if tuple(a.shape) != tuple(shape):
            raise ValueError("{}: '{}' has shape {}, expected {}".format(what, name, tuple(a.shape), tuple(shape)))
        if dtype_name(a) != dtype:
            raise ValueError("{}: '{}' has dtype {}, expected {}".format(what, name, dtype_name(a), dtype))
    for name in got:
        if name not in names:
            raise ValueError("{}: '{}' is not expected here".format(what, name))


def spec(named):
    """[(name, shape, dtype name)] of (name, array) pairs"""
    return [(name, tuple(a.shape), dtype_name(a)) for name, a in named]


def rng_arrays(random_state):
    """A numpy RandomState's state as two arrays: the MT19937 key words and (position, has_gauss, cached_gaussian)."""
    kind, keys, pos, has_gauss, cached = random_state.get_state()
    assert kind == "MT19937"
    return {"rng_keys": np.asarray(keys, np.uint32), "rng_tail": np.array([pos, has_gauss, cached], np.float64)}


def set_rng(random_state, arrays):
    pos, has_gauss, cached = np.asarray(arrays["rng_tail"]).tolist()
    random_state.set_state(("MT19937", np.asarray(arrays["rng_keys"]), int(pos), int(has_gauss), float(cached)))
