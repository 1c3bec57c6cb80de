"""Out-of-bounds WRITE detection without compute-sanitizer (the tool is closed on this GPU pool: profiles/
r02_sanitizer_memcheck.log holds the refusal).  Every kernel family that writes into caller-provided memory gets its
outputs - and, where the entry point takes one, its workspace - carved out of the middle of one arena filled with a
sentinel, with guard bands on both sides and between them, at odd sizes and strided views; after the call every guard
word must still hold the sentinel.  (Reads outside a buffer are not caught this way; the parity tests run every kernel on
ragged sizes whose last tile is partial, where a stray read shows up as a wrong value or an illegal address.)"""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import glorot, random_bipartite

pytestmark = pytest.mark.gpu
SENT = -7.25e30
GUARD = 4096  # floats on each side


class Arena:
    def __init__(self, dev, floats):
        self.buf = torch.full((floats,), SENT, device=dev, dtype=torch.float32)
        self.used = torch.zeros(floats, dtype=torch.bool, device=dev)
        self.off = GUARD

    def take(self, rows, cols, ld=None):
        """[rows, cols] view with leading dimension ld, 32-byte aligned, guard bands around it"""
        ld = ld or cols
        self.off = (self.off + 7) // 8 * 8
        view = self.buf[self.off:self.off + rows * ld].view(rows, ld)[:, :cols]
        self.used[self.off:self.off + rows * ld].view(rows, ld)[:, :cols] = True
        self.off += rows * ld + GUARD
        assert self.off + GUARD <= self.buf.numel()
        return view

    def check(self, what):
        bad = (~self.used) & (self.buf != SENT)
        assert not bool(bad.any()), "%s wrote outside its output: %d stray words, first at %d" % (
            what, int(bad.sum()), int(bad.nonzero()[0]))


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.mark.parametrize("d", [128, 100, 6, 48])
def test_sparse_kernels_stay_inside_their_outputs(dev, d):
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import CsrSlice, DeviceGraph
    adj = random_bipartite(211, 67, 4000, seed=d, n_props=13, n_links=90, dup_links=9)
    n = adj.shape[0]
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=16)
    x = torch.randn(n, d, device=dev)
    for blocking in ((0, 0), (23, 9)):
        norm = CsrSlice(g.norm.rowptr, g.norm.colidx, g.norm.vals, n, 16, blocking=blocking)
        raw = CsrSlice(g.raw.rowptr, g.raw.colidx, None, n, 16, blocking=blocking)
        need = ops.L.load().cbrs_spmm_workspace_bytes(ctypes.byref(norm.desc), d)
        a = Arena(dev, 3 * n * (d + 9) + need // 4 + 8 * GUARD)
        y1, y2 = a.take(n, d, d + 9), a.take(n, d)
        ws = a.take(1, max(need // 4, 1)).view(-1).view(torch.uint8) if need else None
        ops.spmm(norm, x, y1, bias=torch.randn(d, device=dev), relu=True, workspace=ws)
        ops.spmm(raw, x, y2, agg=2, workspace=ws)
        a.check("spmm d=%d blocking=%s" % (d, blocking))
        if d % 2 == 0:
            a = Arena(dev, n * (d + 5) + 4 * GUARD)
            y = a.take(n, d, d + 5)
            ops.gat(raw, x, torch.randn(n, device=dev), torch.randn(n, device=dev), y, bias=torch.randn(d, device=dev))
            a.check("gat d=%d blocking=%s" % (d, blocking))


@pytest.mark.parametrize("m,k,n", [(333, 128, 128), (129, 32, 16), (1000, 64, 256), (1, 96, 48)])
def test_dense_kernels_stay_inside_their_outputs(dev, m, k, n):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(m)
    x, w, b = torch.randn(m, k, device=dev), _t(glorot(rng, (k, n)), dev), torch.randn(n, device=dev)
    a = Arena(dev, 4 * m * (n + 8) + 3 * (m + 50) * n + 16 * GUARD)
    o1, o2, o3 = a.take(m, n, n + 8), a.take(m, n), a.take(m, n, n + 8)
    ops.dense(x, w, b, "relu", out=o1)
    ops.dense_tf32x3(x, w, b, "relu", out=o2)
    ops.dense_tf32x3(x, w, out=o3)
    a.check("dense / dense_tf32x3 %s" % ((m, k, n),))
    if n <= 256 and k % 8 == 0:
        o4 = a.take(m, n, n + 8)
        ops.dense_tc(x, w, b, "relu", out=o4)
        a.check("dense_tc %s" % ((m, k, n),))
    if n <= 128:
        stack = a.take(3 * (m + 50), n)
        ops.dense_grouped(x, [w, w * 0.5, w * 2.0], stack[7:], m + 50)
        for r in range(3):   # the rows between the written blocks are part of the view: they must be untouched too
            blk = stack[r * (m + 50):(r + 1) * (m + 50)]
            assert (blk[:7] == SENT).all() and (blk[7 + m:] == SENT).all()
        a.check("dense_grouped %s" % ((m, k, n),))
