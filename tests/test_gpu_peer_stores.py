"""The multi-GPU exchange, tested on one GPU.

Under the row partition (distributed.py) the producing kernels store every finished row into the local buffer AND into
each peer's copy of it (the *_bcast / *_peers forms), push_rows moves finished blocks, and cbrs_peer_barrier
orders producers before consumers.  Every peer store is a plain store to an address the caller supplies, so a separate
allocation on the same device stands in for another rank's copy and nothing in the kernel changes but the address.

A. Kernel by kernel: the same call without peers, then with 1 and with 7 (CBRS_MAX_PEERS - 1) stand-in copies carved
   from one sentinel-filled arena with guard bands between them.  The local output must keep its bits, every copy must
   hold the same bits, and every word outside the views must still hold the sentinel.  A copy has the local output's
   layout (same leading dimension and alignment, as every rank's copy of a symmetric buffer has); the layouts used are
   packed rows, column slices of wider rows and rows that start off a 16-byte boundary.  The entry points must also
   refuse peer lists they cannot serve, before any launch.
B. SymmetricBuffer addresses and push_rows (vector and scalar paths, the multicast target).
C. The flag barrier, only in configurations where every flag it waits for is already set: the kernel traps when a
   peer does not arrive, so no configuration that could make it wait is run.
D. A loopback of the partitioned layer loop: RowPartition.propagate itself on 2 and 3 ranks emulated by threads of one
   process, all launching on one stream, over an emulated heap of symmetric buffers and a host-side barrier.  Every
   rank's result, with every layer's output concatenated, must equal the single-GPU SequentialGNN result bit for bit,
   on the first call and on a second that reuses the buffers - the claim selfcheck.partition_parity makes on several
   GPUs."""
import ctypes
import threading
import types

import numpy as np
import pytest
import torch

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import assert_close, random_bipartite

pytestmark = pytest.mark.gpu
SENT = -7.25e30
GUARD = 1024        # float words between and around the views
MAX_COPIES = 7      # CBRS_MAX_PEERS - 1
F32, BF16 = torch.float32, torch.bfloat16


class Arena:
    """One sentinel-filled float32 allocation from which output views are carved with guard bands around them."""

    def __init__(self, dev, words):
        self.buf = torch.full((int(words),), SENT, dtype=F32, device=dev)
        self.used = torch.zeros(int(words), dtype=torch.bool, device=dev)
        self.off = GUARD

    @staticmethod
    def words(rows, ld, dtype=F32, shift=0):
        per = 2 if dtype == BF16 else 1
        return -(-(shift + rows * ld) // per) + 8 + GUARD

    def take(self, rows, cols, ld=None, dtype=F32, shift=0, mark=True):
        """[rows, cols] view with leading dimension ld (elements) that starts `shift` elements past a 32-byte boundary"""
        ld = ld or cols
        per = 2 if dtype == BF16 else 1
        words = -(-(shift + rows * ld) // per)
        self.off = (self.off + 7) // 8 * 8
        assert self.off + words + GUARD <= self.buf.numel(), "arena too small"
        flat = self.buf[self.off:self.off + words]
        if dtype == BF16:
            flat = flat.view(BF16)
        view = flat[shift:shift + rows * ld].view(rows, ld)[:, :cols]
        if mark and rows and cols:
            idx = shift + torch.arange(rows, device=self.buf.device)[:, None] * ld + torch.arange(cols, device=self.buf.device)
            self.used[self.off + idx.reshape(-1) // per] = True
        self.off += words + GUARD
        return view

    def mark(self, view):
        """an fp32 view of the arena that a call is allowed to write"""
        if view.numel():
            off = (view.data_ptr() - self.buf.data_ptr()) // 4
            torch.as_strided(self.used, view.shape, view.stride(), off).fill_(True)

    def check(self, what):
        bad = (~self.used) & (self.buf != SENT)
        assert not bool(bad.any()), "%s wrote outside its output: %d stray words, first at %d" % (
            what, int(bad.sum()), int(bad.nonzero()[0]))


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _sentinel_rows(rows, cols, dtype):
    s = torch.full((2,), SENT, dtype=F32).view(dtype) if dtype == BF16 else torch.full((1,), SENT, dtype=F32)
    return s.repeat(cols // s.numel()).expand(rows, cols)


def check_peer_stores(dev, specs, run, what, counts=(1, MAX_COPIES), peer_shift=None, local_bits=True):
    """specs: one (rows, cols, ld, dtype, shift) per output that the entry point also stores into every copy (out; q).
    run(views, peers) launches on the local views; peers is None or, per output, the addresses of its copies.
    peer_shift(i): shift of copy i when it differs from the local output's.  Returns (views of the run without peers,
    local views of the run with the most copies)."""
    def carve(n_copies):
        words = 2 * GUARD + sum(Arena.words(r, ld, dt, max(sh, 8)) for r, _, ld, dt, sh in specs) * (1 + n_copies)
        a = Arena(dev, words)
        local = [a.take(r, c, ld, dt, sh) for r, c, ld, dt, sh in specs]
        copies = [[a.take(r, c, ld, dt, peer_shift(i) if peer_shift else sh) for i in range(n_copies)]
                  for r, c, ld, dt, sh in specs]
        return a, local, copies

    a0, ref, _ = carve(0)
    run(ref, None)
    torch.cuda.synchronize()
    a0.check(what + " without peers")
    local = ref
    for k in counts:
        a, local, copies = carve(k)
        run(local, [[c.data_ptr() for c in cs] for cs in copies])
        torch.cuda.synchronize()
        a.check("%s with %d peer copies" % (what, k))
        for s, (lv, rv, cs) in enumerate(zip(local, ref, copies)):
            if local_bits:
                assert same_bits(lv, rv), "%s: %d peer copies changed the bits of local output %d" % (what, k, s)
            for i, c in enumerate(cs):
                assert same_bits(c, lv), "%s: copy %d of %d of output %d differs from the local output" % (what, i, k, s)
    return ref, local


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def graph(dev):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(211, 67, 4000, seed=3, n_props=13, n_links=90, dup_links=9)
    return adj, DeviceGraph.from_scipy(adj, dev, chunk_edges=16)


def _sched(g, view, blocking, chunk_edges=16):
    from deep_cbrs_amar_renaissance_b200.graph import CsrSlice
    v = getattr(g, view)
    return CsrSlice(v.rowptr, v.colidx, v.vals, v.n_cols, chunk_edges, blocking=blocking)


def _heavy_row(csr, min_len=25):
    """a row of at least min_len edges (split into chunks, and column-blocked under blocking=(*, <= min_len)) in the
    middle of the rows past the first third"""
    lens = (csr.rowptr[1:] - csr.rowptr[:-1]).cpu().numpy()
    rows = np.nonzero(lens >= min_len)[0]
    rows = rows[rows >= len(lens) // 3]
    return int(rows[len(rows) // 2])


def _randn(shape, dev, seed, scale=1.0):
    return torch.randn(*shape, device=dev, generator=torch.Generator(dev).manual_seed(seed)) * scale


def _code(code):
    return pytest.raises(RuntimeError, match=r"\(code %d\)" % code)


# ----------------------------------------------------------------------------------------------------- A. SpMM
SPMM_SOURCES = [(F32, 48), (F32, 128), (F32, 6), (F32, 130), (BF16, 128), (BF16, 12), (BF16, 7)]   # VEC 4, 4, 1, 1 | 8, 4, 1


@pytest.mark.parametrize("blocking", [(0, 0), (23, 9)])
@pytest.mark.parametrize("xdt,d", SPMM_SOURCES)
def test_spmm_peer_stores(dev, graph, xdt, d, blocking):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj, g = graph
    n = adj.shape[0]
    x = _randn((n, d), dev, d).to(xdt)
    bias = _randn((d,), dev, d + 1)
    # row-major: packed rows; blocked: a column slice of wider rows, 16 bytes in
    ld, shift = (d, 0) if blocking == (0, 0) else (d + 8, 4)
    xs = x.float().cpu().numpy().astype(np.float64)
    ptr, idx, _ = og.reorder_raw(adj)
    for view, agg, kw, want in (("norm", 0, dict(bias=bias, relu=True),
                                 np.maximum(og.gcn_filter(adj) @ xs + bias.cpu().numpy(), 0)),
                                ("raw", 1, {}, ol.sage_aggregate(xs, ptr, idx, "sum")),
                                ("raw", 2, {}, ol.sage_aggregate(xs, ptr, idx, "mean"))):
        csr = _sched(g, view, blocking)
        assert csr.chunks["n_heavy"] > 0          # the heavy-row kernel stores too

        def run(v, peers):
            ops.spmm(csr, x, v[0], agg=agg, peers=peers[0] if peers else None, **kw)
        what = "spmm %s d=%d agg=%d blocking=%s" % (xdt, d, agg, blocking)
        ref, _ = check_peer_stores(dev, [(n, d, ld, F32, shift)], run, what)
        assert_close(ref[0].cpu().numpy(), want, what=what)


@pytest.mark.parametrize("blocking", [(0, 0), (23, 9)])
def test_spmm_misaligned_peer_drops_to_scalar_stores(dev, graph, blocking):
    """one copy 4 bytes off a 16-byte boundary: the kernel must take its VEC 1 form for every copy"""
    from deep_cbrs_amar_renaissance_b200 import ops
    adj, g = graph
    n, d = adj.shape[0], 128
    x, bias = _randn((n, d), dev, 5), _randn((d,), dev, 6)
    csr = _sched(g, "norm", blocking)

    def run(v, peers):
        ops.spmm(csr, x, v[0], bias=bias, relu=True, peers=peers[0] if peers else None)
    _, local = check_peer_stores(dev, [(n, d, d, F32, 0)], run, "spmm misaligned peer",
                                 peer_shift=lambda i: 1 if i == 0 else 0, local_bits=False)
    want = np.maximum(og.gcn_filter(adj) @ x.cpu().numpy().astype(np.float64) + bias.cpu().numpy(), 0)
    assert_close(local[0].cpu().numpy(), want, what="spmm with a misaligned peer")


@pytest.mark.parametrize("blocking", [(0, 0), (23, 9)])
@pytest.mark.parametrize("h", [8, 20, 128])
def test_gat_peer_stores(dev, graph, h, blocking):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj, g = graph
    n = adj.shape[0]
    csr = _sched(g, "raw", blocking)
    z, p, q, bias = _randn((n, h), dev, h), _randn((n,), dev, h + 1), _randn((n,), dev, h + 2), _randn((h,), dev, h + 3)
    full = torch.empty(n, h, device=dev)
    ops.gat(csr, z, p, q, full, bias=bias, relu=True)
    hv = _heavy_row(csr)
    for r0, r1, ld, shift in ((0, n, h, 0), (hv, n - 17, h + 3, 1)):    # a slice that starts at a heavy row
        sl = csr if (r0, r1) == (0, n) else csr.row_slice(r0, r1)
        assert sl.chunks["n_heavy"] > 0

        def run(v, peers):
            ops.gat(sl, z, p, q, v[0], bias=bias, relu=True, row_offset=r0, peers=peers[0] if peers else None)
        ref, _ = check_peer_stores(dev, [(r1 - r0, h, ld, F32, shift)], run,
                                   "gat h=%d rows %d:%d blocking=%s" % (h, r0, r1, blocking))
        assert same_bits(ref[0], full[r0:r1])


# ----------------------------------------------------------------------------------------------------- A. dense
# (name, m, f1, f2, n, gathered, rowop, act, out dtype, leading-dimension pad, shift)
DENSE_CASES = [
    ("tiled", 333, 24, 0, 20, False, 0, "relu", F32, 3, 1),
    ("fast", 333, 64, 0, 64, False, 0, "relu", F32, 8, 4),
    ("fast-scalar-stores", 200, 32, 0, 128, False, 0, "sigmoid", F32, 1, 1),
    ("gather-concat-fast", 257, 32, 16, 48, True, 0, "tanh", F32, 0, 0),
    ("gather-concat-tiled", 257, 32, 16, 20, True, 0, None, F32, 4, 4),
    ("attn-fast", 301, 64, 0, 32, False, 2, None, F32, 8, 4),
    ("attn-tiled", 301, 24, 0, 20, False, 2, None, F32, 0, 0),
    ("l2norm-fast", 290, 32, 32, 48, False, 1, "relu", F32, 4, 4),
    ("l2norm-tiled", 290, 24, 24, 20, False, 1, "relu", F32, 0, 0),
    ("l2norm-128", 290, 64, 64, 128, True, 1, "relu", F32, 0, 0),
    ("bf16-fast", 333, 64, 0, 64, False, 0, "relu", BF16, 8, 4),
    ("bf16-fast-gather", 129, 32, 16, 96, True, 0, None, BF16, 0, 0),
    ("bf16-tiled", 333, 24, 0, 20, False, 0, "relu", BF16, 2, 2),
]


@pytest.mark.parametrize("case", DENSE_CASES, ids=[c[0] for c in DENSE_CASES])
def test_dense_peer_stores(dev, case):
    from deep_cbrs_amar_renaissance_b200 import ops
    name, m, f1, f2, n, gathered, rowop, act, odt, pad, shift = case
    rows1, rows2 = m + 41, m + 7
    x1 = _randn((rows1 if gathered else m, f1), dev, 1)
    x2 = _randn((rows2 if gathered else m, f2), dev, 2) if f2 else None
    idx1 = torch.randint(0, rows1, (m,), device=dev, generator=torch.Generator(dev).manual_seed(3)) if gathered else None
    idx2 = torch.randint(0, rows2, (m,), device=dev, generator=torch.Generator(dev).manual_seed(4)) if gathered and f2 else None
    w = _randn((f1 + f2, n), dev, 5, (f1 + f2) ** -0.5)
    b = _randn((n,), dev, 6, 0.1)
    a_s, a_n = (_randn((n,), dev, 7), _randn((n,), dev, 8)) if rowop == 2 else (None, None)
    specs = [(m, n, n + pad, odt, shift)] + ([(m, 1, 1, F32, 0)] if rowop == 2 else [])

    def run(v, peers):
        ops.dense(x1, w, b, act, x2=x2, idx1=idx1, idx2=idx2, rowop=rowop, a_self=a_s, a_neigh=a_n, out=v[0],
                  q_out=v[1].view(-1) if rowop == 2 else None, peers=peers[0] if peers else None,
                  q_peers=peers[1] if peers and rowop == 2 else None)
    ref, _ = check_peer_stores(dev, specs, run, "dense " + name)
    # the run without peers against float64
    xs = x1[idx1] if gathered else x1
    if f2:
        xs = torch.cat([xs, x2[idx2] if gathered else x2], 1)
    v = xs.double().cpu().numpy() @ w.double().cpu().numpy() + b.double().cpu().numpy()
    if rowop == 1:
        v = v / np.sqrt(np.maximum((v * v).sum(1, keepdims=True), 1e-12))
    if rowop == 2:
        assert_close(ref[1].view(-1).cpu().numpy(), v @ a_n.double().cpu().numpy(), what=name + " q")
    v = {None: v, "relu": np.maximum(v, 0), "tanh": np.tanh(v), "sigmoid": 1 / (1 + np.exp(-v))}[act]
    if odt == BF16:
        out32 = ops.dense(x1, w, b, act, x2=x2, idx1=idx1, idx2=idx2, rowop=rowop, a_self=a_s, a_neigh=a_n)
        assert same_bits(ref[0], out32.to(BF16))    # the fp32 result rounded to nearest even
    else:
        assert_close(ref[0].cpu().numpy(), v, what=name)


@pytest.mark.parametrize("odt", [F32, BF16])
def test_dense_grouped_peer_stores(dev, odt):
    """a row-offset view of the stacked relational operand: in every copy the rows between relation blocks stay as
    they were"""
    from deep_cbrs_amar_renaissance_b200 import ops
    m, f, h, R, G, a = 150, 64, 32, 3, 170, 11
    x = _randn((m, f), dev, 1)
    kernels = [_randn((f, h), dev, 2 + r, 0.125) for r in range(R)]

    def run(v, peers):
        st = v[0][a:]
        off = st.data_ptr() - v[0].data_ptr()
        ops.dense_grouped(x, kernels, st, G, peers=[p + off for p in peers[0]] if peers else None)
    ref, local = check_peer_stores(dev, [(R * G, h, h, odt, 0)], run, "dense_grouped %s" % odt)
    for stack in (ref[0], local[0]):
        for r in range(R):
            blk = stack[r * G:(r + 1) * G]
            assert same_bits(blk[:a], _sentinel_rows(a, h, odt).to(dev))
            assert same_bits(blk[a + m:], _sentinel_rows(G - a - m, h, odt).to(dev))
            want = x.double() @ kernels[r].double()
            assert_close(blk[a:a + m].float().cpu().numpy(), want.cpu().numpy(), rtol=1e-5 if odt == F32 else 1e-2)


# (name, m, k, n, out dtype, leading-dimension pad, shift): 8-wide stores, scalar stores, bf16 stores
TF32_CASES = [("f32-v8", 333, 64, 64, F32, 0, 0), ("f32-scalar", 333, 64, 48, F32, 4, 4), ("bf16", 333, 128, 128, BF16, 16, 0)]


@pytest.mark.parametrize("case", TF32_CASES, ids=[c[0] for c in TF32_CASES])
def test_tf32x3_transform_peer_stores(dev, case):
    from deep_cbrs_amar_renaissance_b200 import ops
    name, m, k, n, odt, pad, shift = case
    x, w, b = _randn((m, k), dev, 1), _randn((k, n), dev, 2, k ** -0.5), _randn((n,), dev, 3)
    want = x.double() @ w.double()
    big = 1 << 16                           # a graph this large takes the tensor-core kernel

    def gcn(v, peers):
        assert ops.tf32x3_chosen(big, k, n, x, v[0])
        ops.gcn_transform(x, w, big, out=v[0], peers=peers[0] if peers else None)

    def biased(v, peers):
        ops.dense_tf32x3(x, w, b, "relu", out=v[0], peers=peers[0] if peers else None)
    for what, run, exp in (("gcn_transform", gcn, want), ("dense_tf32x3 bias relu", biased, torch.relu(want + b.double()))):
        ref, _ = check_peer_stores(dev, [(m, n, n + pad, odt, shift)], run, "%s %s" % (what, name))
        if odt == F32:
            assert_close(ref[0].cpu().numpy(), exp.cpu().numpy(), what=what)
        else:
            full = torch.empty(m, n, device=dev)
            (gcn if run is gcn else biased)([full], None)
            assert same_bits(ref[0], full.to(BF16))


def test_tf32x3_attention_and_graphsage_peer_stores(dev):
    """gat_transform with q_peers (cbrs_dense_tf32x3_attn) and sage_dense's second product (cbrs_dense_tf32x3_ex)"""
    from deep_cbrs_amar_renaissance_b200 import ops
    m, k, n = 333, 64, 64
    big = 1 << 16
    x, w = _randn((m, k), dev, 1), _randn((k, n), dev, 2, k ** -0.5)
    a_s, a_n = _randn((n,), dev, 3), _randn((n,), dev, 4)

    def attn(v, peers):
        assert ops.tf32x3_chosen(big, k, n, x, v[0])
        ops.gat_transform(x, w, a_s, a_n, big, out=v[0], q_out=v[1].view(-1), peers=peers[0] if peers else None,
                          q_peers=peers[1] if peers else None)
    ref, _ = check_peer_stores(dev, [(m, n, n + 4, F32, 4), (m, 1, 1, F32, 0)], attn, "gat_transform tf32x3")
    z64 = x.double() @ w.double()
    assert_close(ref[0].cpu().numpy(), z64.cpu().numpy(), what="z")
    assert_close(ref[1].view(-1).cpu().numpy(), (z64 @ a_n.double()).cpu().numpy(), what="q")

    f, n = 64, 48
    xs, agg = _randn((m, f), dev, 5), _randn((m, f), dev, 6)
    kern, b = _randn((2 * f, n), dev, 7, 0.1), _randn((n,), dev, 8, 0.1)

    def sage(v, peers):
        assert ops.tf32x3_chosen(big, f, n, xs, v[0]) and ops.tf32x3_chosen(big, f, n, agg)
        ops.sage_dense(xs, agg, kern, b, "relu", big, out=v[0], peers=peers[0] if peers else None)
    ref, _ = check_peer_stores(dev, [(m, n, n + 8, F32, 0)], sage, "sage_dense tf32x3")
    v = torch.cat([xs, agg], 1).double() @ kern.double() + b.double()
    want = torch.relu(v / v.norm(dim=1, keepdim=True).clamp_min(1e-6))
    assert_close(ref[0].cpu().numpy(), want.cpu().numpy(), what="sage_dense")


def test_peer_lists_the_kernels_cannot_serve_are_refused_before_any_launch(dev, graph):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj, g = graph
    n = adj.shape[0]
    csr = _sched(g, "norm", (0, 0))
    a = Arena(dev, 2 * GUARD + 12 * Arena.words(n, 160))
    out = a.take(n, 128)
    copies = [a.take(n, 128).data_ptr() for _ in range(8)]
    out160, copy160 = a.take(n, 160), a.take(n, 160).data_ptr()
    x, w, b = _randn((n, 128), dev, 1), _randn((128, 128), dev, 2, 0.1), _randn((128,), dev, 3)
    p, q, a_s, a_n = _randn((n,), dev, 4), _randn((n,), dev, 5), _randn((128,), dev, 6), _randn((128,), dev, 7)
    w160 = _randn((128, 160), dev, 8, 0.1)
    bf = a.take(n, 128, 128, BF16)
    bf_copy = a.take(n, 128, 128, BF16).data_ptr()
    torch.cuda.synchronize()
    E_INVALID, E_UNSUPPORTED = -1, -4
    cases = [
        ("spmm, 8 peers", E_INVALID, lambda: ops.spmm(csr, x, out, peers=copies)),
        ("spmm, a null peer", E_INVALID, lambda: ops.spmm(csr, x, out, peers=[copies[0], 0])),
        ("gat, 8 peers", E_INVALID, lambda: ops.gat(g.raw, x, p, q, out, peers=copies)),
        ("gat, a null peer", E_INVALID, lambda: ops.gat(g.raw, x, p, q, out, peers=[0])),
        ("dense, 8 peers", E_INVALID, lambda: ops.dense(x, w, b, out=out, peers=copies)),
        ("dense, a null peer", E_INVALID, lambda: ops.dense(x, w, b, out=out, peers=[copies[0], 0])),
        ("dense, peer aligned differently mod 16", E_INVALID, lambda: ops.dense(x, w, b, out=out, peers=[copies[0] + 4])),
        ("dense bf16, peer aligned differently mod 16", E_INVALID,
         lambda: ops.dense(x, w, b, out=bf, peers=[bf_copy + 8])),
        ("dense attention, peers but no q_peers", E_INVALID,
         lambda: ops.dense(x, w, rowop=2, a_self=a_s, a_neigh=a_n, out=out, peers=[copies[0]])),
        ("dense l2norm n > 128 with peers", E_UNSUPPORTED,
         lambda: ops.dense(x, w160, rowop=1, out=out160, peers=[copy160])),
        ("dense_grouped, 8 peers", E_INVALID, lambda: ops.dense_grouped(x[:50], [w[:, :64], w[:, 64:]], out[:, :64], 60,
                                                                          peers=copies)),
        ("dense_tf32x3, 8 peers", E_INVALID, lambda: ops.dense_tf32x3(x, w, out=out, peers=copies)),
        ("dense_tf32x3, a null peer", E_INVALID, lambda: ops.dense_tf32x3(x, w, out=out, peers=[0])),
        ("dense_tf32x3, peer aligned differently mod 32", E_INVALID,
         lambda: ops.dense_tf32x3(x, w, out=out, peers=[copies[0] + 16])),
        ("dense_tf32x3 bf16, peer aligned differently mod 32", E_INVALID,
         lambda: ops.dense_tf32x3(x, w, out=bf, peers=[bf_copy + 16])),
        ("gat_transform tf32x3, peers but no q_peers", E_INVALID,
         lambda: ops.gat_transform(x, w, a_s, a_n, 1 << 16, out=out, peers=[copies[0]])),
        ("sage_dense tf32x3, 8 peers", E_INVALID,
         lambda: ops.sage_dense(x[:, :64], x[:, 64:], w, b, "relu", 1 << 16, out=out, peers=copies)),
    ]
    for what, code, call in cases:
        with _code(code):
            call()
        torch.cuda.synchronize()
        assert bool((a.buf == SENT).all()), what + ": refused, but something was written"


# ------------------------------------------------------------------------------------- B. addresses and pushes
def _stub(rank):
    return types.SimpleNamespace(rank=rank)


@pytest.mark.parametrize("world", [2, 8])
def test_symmetric_buffer_addresses(dev, world):
    from deep_cbrs_amar_renaissance_b200.distributed import SymmetricBuffer
    nbytes = 4096 * 4
    copies = [torch.empty(nbytes // 4, device=dev) for _ in range(world)]
    ptrs = [c.data_ptr() for c in copies]
    mc = torch.empty(nbytes // 4, device=dev)
    for rank in sorted({0, 1, world - 1}):
        sb = SymmetricBuffer(_stub(rank), nbytes, ptrs)
        sbm = SymmetricBuffer(_stub(rank), nbytes, ptrs, mc_ptr=mc.data_ptr())
        assert sb.local == ptrs[rank] and sb.flat.data_ptr() == ptrs[rank] and sb.flat.numel() == nbytes // 4
        m = sb.matrix(100, 40)
        for view in (m, m[7:19], m[7:19, 3:11], m[99:100, 39], m[:, 5], sb.matrix(200, 20, torch.bfloat16)[5:9, 1:3],
                     sb.flat[nbytes // 4 - 1:]):
            off = view.data_ptr() - ptrs[rank]
            assert sb.peer_addrs(view) == [p + off for r, p in enumerate(ptrs) if r != rank]
            assert sb.mc_addr(view) is None and sbm.mc_addr(view) == mc.data_ptr() + off
        for outside in (copies[(rank + 1) % world][:4], mc[:4]):
            with pytest.raises(ValueError):
                sb.peer_addrs(outside)
            with pytest.raises(ValueError):
                sbm.mc_addr(outside)


N_PUSH, W_PUSH = 64, 16
PUSH_VIEWS = {   # a view of one rank's copy (a flat float tensor), selected the same way in every copy
    "float4": lambda f: f[:N_PUSH * 8].view(N_PUSH, 8)[5:41],
    "q column (w=1)": lambda f: f[:N_PUSH].view(N_PUSH, 1)[3:50, 0],
    "w=6": lambda f: f[:N_PUSH * 6].view(N_PUSH, 6)[2:33],
    "misaligned": lambda f: f[:N_PUSH * 8].view(N_PUSH, 8)[4:20, 1:5],
    "column slice": lambda f: f[:N_PUSH * W_PUSH].view(N_PUSH, W_PUSH)[9:30, 4:12],
    "m=1": lambda f: f[:N_PUSH * W_PUSH].view(N_PUSH, W_PUSH)[17:18, 4:12],
    "m=0": lambda f: f[:N_PUSH * W_PUSH].view(N_PUSH, W_PUSH)[17:17],
    "m=0 at the end": lambda f: f[:N_PUSH * W_PUSH].view(N_PUSH, W_PUSH)[N_PUSH:],
}


@pytest.mark.parametrize("multicast", [False, True])
@pytest.mark.parametrize("name", list(PUSH_VIEWS))
def test_push_rows(dev, name, multicast):
    """every other rank's copy (or, with a multicast mapping, only that address) receives exactly the view"""
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.distributed import SymmetricBuffer
    world, rank, words = 3, 1, N_PUSH * W_PUSH
    a = Arena(dev, 2 * GUARD + (world + 1) * (words + 8 + GUARD))
    flats = [a.take(1, words, mark=(r == rank)).view(-1) for r in range(world + 1)]   # the last one: a multicast target
    flats[rank].copy_(_randn((words,), dev, 9))
    before = flats[rank].clone()
    sb = SymmetricBuffer(_stub(rank), words * 4, [f.data_ptr() for f in flats[:world]],
                         mc_ptr=flats[world].data_ptr() if multicast else 0)
    sel = PUSH_VIEWS[name]
    view = sel(flats[rank])
    launches = ops.LAUNCHES
    ops.push_rows(view, sb)
    torch.cuda.synchronize()
    assert ops.LAUNCHES - launches == (0 if view.numel() == 0 else 1 if multicast else world - 1)
    targets = [world] if multicast else [r for r in range(world) if r != rank]
    for r in targets:
        assert same_bits(sel(flats[r]), view), "%s: copy %d" % (name, r)
        a.mark(sel(flats[r]))
    assert same_bits(flats[rank], before)
    a.check("push_rows %s%s" % (name, " (multicast)" if multicast else ""))


# ----------------------------------------------------------------------------------------------- C. the flag barrier
@pytest.mark.parametrize("n_ranks,me", [(1, 0), (2, 0), (2, 1), (8, 0), (8, 5)])
def test_flag_barrier_publishes_its_epoch(dev, n_ranks, me):
    """Every other rank has already published the epoch into this rank's array, so the kernel never waits: it must
    publish the epoch at slot `me` of every rank's array, touch nothing else and leave status 0."""
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    lib = L.load()
    flags = torch.zeros(n_ranks, L.MAX_PEERS, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    arr = (ctypes.c_void_p * n_ranks)(*[flags[r].data_ptr() for r in range(n_ranks)])
    for epoch in (1, 2, 7):
        flags[me, :n_ranks] = epoch
        flags[me, me] = epoch - 1                    # this rank's own slot is written by the launch itself
        torch.cuda.synchronize()
        pre = flags.cpu()
        # the kernel spins until flags[me][t] >= epoch for every t: all but its own slot must hold already
        assert all(int(pre[me, t]) >= epoch for t in range(n_ranks) if t != me)
        L.check(lib.cbrs_peer_barrier(arr, n_ranks, me, epoch, ctypes.c_void_p(status.data_ptr()), 30.0, stream),
                "cbrs_peer_barrier")
        torch.cuda.synchronize()
        want = pre.clone()
        want[:, me] = epoch
        assert torch.equal(flags.cpu(), want) and int(status.item()) == 0
    # refused on the host.  Only arguments that could neither wait nor fault if a launch did happen: epoch 0 is
    # reached at once, and a launch would be seen as zeros written into the flags
    st = ctypes.c_void_p(status.data_ptr())
    assert lib.cbrs_peer_barrier(arr, 0, 0, 0, st, 30.0, stream) == -1
    assert lib.cbrs_peer_barrier(arr, n_ranks, me, 0, None, 30.0, stream) == -1
    assert lib.cbrs_peer_barrier(None, n_ranks, me, 0, st, 30.0, stream) == -1
    torch.cuda.synchronize()
    assert torch.equal(flags.cpu(), want) and int(status.item()) == 0


# ------------------------------------------------------------------------- D. loopback of the partitioned layer loop
class _Heap:
    """What the peer layer loop uses of a PeerHeap, for one of `world` ranks emulated by threads of this process.
    alloc() is collective, as PeerHeap.alloc is: the k-th call of every rank returns a SymmetricBuffer over the same
    `world` sentinel-filled allocations.  barrier() is a host-side rendezvous of the threads.  Every thread launches on
    one stream, so when the rendezvous opens, every rank's earlier launches are queued ahead of every rank's later
    ones: the ordering the flag barrier gives across GPUs."""

    def __init__(self, shared, rank):
        self.shared, self.rank, self.n_allocs = shared, rank, 0

    def alloc(self, nbytes):
        from deep_cbrs_amar_renaissance_b200.distributed import SymmetricBuffer
        nbytes = (int(nbytes) + 255) // 256 * 256
        sh = self.shared
        with sh.lock:
            if self.n_allocs == len(sh.allocs):
                sh.allocs.append((nbytes, [torch.full((nbytes // 4,), SENT, device=sh.dev) for _ in range(sh.world)]))
            size, copies = sh.allocs[self.n_allocs]
        self.n_allocs += 1
        assert size == nbytes, "rank %d asked for %d bytes, another rank for %d" % (self.rank, nbytes, size)
        return SymmetricBuffer(self, nbytes, [c.data_ptr() for c in copies])

    def barrier(self):
        self.shared.rendezvous.wait()


def _ranks(sizes, cuts, dev):
    """One RowPartition per emulated rank, rank r owning rows cuts[r]:cuts[r+1], with the attributes
    RowPartition.__init__ sets that the peer layer loop reads.  Every node type is final, so every rank ends up with
    every row."""
    from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
    world = len(cuts) - 1
    shared = types.SimpleNamespace(world=world, dev=dev, lock=threading.Lock(), allocs=[],
                                   rendezvous=threading.Barrier(world, timeout=120))
    parts = []
    for r in range(world):
        p = RowPartition.__new__(RowPartition)
        p.group, p.exchange, p.heap = None, "peer", _Heap(shared, r)
        p.n_rows_by_type, p.world, p.rank = list(sizes), world, r
        p.mine = [(cuts[r], cuts[r + 1])]
        p.final_types = list(range(len(sizes)))
        p._sym, p._slices, p._bufs = {}, {}, {}
        parts.append(p)
    return shared, parts


def _propagate_on_every_rank(shared, parts, seq, calls=2):
    """RowPartition.propagate `calls` times on every emulated rank, each rank in its own thread, all on the caller's
    stream -> [[copy of the result of each call] per rank].  A rank that raises breaks the rendezvous, so the others
    stop waiting for it, and its error is raised here."""
    stream = torch.cuda.current_stream()
    results = [[] for _ in parts]
    errors = [None] * len(parts)

    def run(r):
        try:
            with torch.cuda.stream(stream):
                for _ in range(calls):
                    results[r].append(parts[r].propagate(seq).clone())
        except BaseException as e:  # noqa: BLE001
            errors[r] = e
            shared.rendezvous.abort()
    threads = [threading.Thread(target=run, args=(r,)) for r in range(len(parts))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    raised = [e for e in errors if e is not None]
    if raised:
        raise next((e for e in raised if not isinstance(e, threading.BrokenBarrierError)), raised[0])
    torch.cuda.synchronize()
    return results


# (family, variant, transform, dtype).  Variants: "64-32-48" = GCN layers of those widths, "2rel" / "1rel" = RGCN with
# that many relations (one relation: the tensor-core transform, which GCNConv would take at this width, is forced)
LOOPBACK = [("gcn", "replicate", t, dt) for t in ("ffma", "tf32x3") for dt in ("fp32", "bf16")]
LOOPBACK += [("gcn", "64-32-48", "ffma", "fp32"), ("rgcn", "2rel", "-", "fp32"), ("rgcn", "1rel", "tf32x3", "fp32")]
LOOPBACK += [(f, "-", t, "fp32") for f in ("gat", "sage") for t in ("ffma", "tf32x3")] + [("lightgcn", "-", "-", "fp32")]


def _stack(family, variant, dtype, g, emb):
    """a three-layer SequentialGNN of `family` over g with the embedding table emb, concatenating every layer's output"""
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.layers import GATConv, GCNConv, GraphSageConv, LightGCNConv, RGCNConv
    from deep_cbrs_amar_renaissance_b200.models.gnn import SequentialGNN
    set_seed(23)
    make = {"gcn": lambda w: GCNConv(w, activation="relu"),
            "rgcn": lambda w: RGCNConv(w, 2 if variant == "2rel" else 1, activation="relu"),
            "gat": lambda w: GATConv(w, activation="relu", dropout_rate=0.0),
            "sage": lambda w: GraphSageConv(w, activation="relu"), "lightgcn": lambda w: LightGCNConv()}[family]
    widths = [64, 32, 48] if variant == "64-32-48" else [emb.shape[1]] * 3
    seq = SequentialGNN(g, [make(w) for w in widths], embedding_dim=emb.shape[1], final_node="concatenation")
    seq.build_layers()
    with torch.no_grad():
        seq.embeddings.copy_(emb)
        for l, ly in enumerate(seq.seq_layers):
            if getattr(ly, "bias", None) is not None:
                ly.bias.copy_(_randn(ly.bias.shape, emb.device, 30 + l, 0.1))
    if dtype == "bf16":
        seq.set_feature_dtype("bf16")
    return seq


@pytest.fixture(scope="module")
def loopback_adj():
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    return small_graph(300, 200, 6000, seed=5, n_props=50, n_links=600, dup_links=40), (300, 200, 50)


@pytest.mark.parametrize("blocked", [False, True], ids=["row-major", "blocked"])
@pytest.mark.parametrize("family,variant,transform,dtype", LOOPBACK, ids=["-".join(c) for c in LOOPBACK])
def test_partitioned_layer_loop_loopback(dev, loopback_adj, monkeypatch, family, variant, transform, dtype, blocked):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200 import ops
    adj, sizes = loopback_adj
    n = adj.shape[0]
    monkeypatch.setattr(G, "FORCED_BLOCKING", (97, 25) if blocked else None)
    if transform != "-":
        monkeypatch.setattr(ops, "GCN_TRANSFORM", transform)
    if variant == "2rel":         # item <-> property links are relation 1 (tests/helpers.relation_blocks)
        rel = ((adj.row >= sizes[0] + sizes[1]) | (adj.col >= sizes[0] + sizes[1])).astype(np.int32)

        def t(v, dt):
            return torch.from_numpy(np.ascontiguousarray(v, dt)).to(dev)
        g = G.DeviceGraph(t(adj.row, np.int32), t(adj.col, np.int32), t(adj.data, np.float32), n, 16, rel=t(rel, np.int32),
                          n_rel=2)
    else:
        g = G.DeviceGraph.from_scipy(adj, dev, chunk_edges=16)
    emb = _randn((n, 128 if family == "gcn" else 64), dev, 11)
    if variant == "1rel":
        assert ops.tf32x3_chosen(n, 64, 64, emb)
    seq = _stack(family, variant, dtype, g, emb)
    full = g.raw if family in ("gat", "sage") else g.norm    # built before the threads start, which only read it
    assert full.blocking == ((97, 25) if blocked else (0, 0)) and full.chunks["n_heavy"] > 0
    ref = seq.call(None).clone()  # the single-GPU layer loop
    L.load()
    hv = _heavy_row(full)
    for cuts in ([0, hv, n], [0, 37, hv + 1, n]):     # uneven cuts; a rank starts, or ends, at a heavy row
        shared, parts = _ranks(sizes, cuts, dev)
        for r, got in enumerate(_propagate_on_every_rank(shared, parts, seq)):
            for k, out in enumerate(got):
                assert same_bits(out, ref), "%s %s %s %s: call %d, rank %d of %d (cuts %s)" % (
                    family, variant, transform, dtype, k, r, len(cuts) - 1, cuts)
