"""The 3xTF32 transform (cbrs_dense_tf32x3 and its _ex / _attn variants) at every width it accepts, on both TMEM
accumulator buffers and with every epilogue, against float64.

The kernel is persistent: CTA c runs tiles c, c + 148, c + 296, ... and the tile with index lt within its CTA
accumulates in TMEM buffer lt % acc_bufs (acc_bufs = 2 when 2 n + 128 <= 512 columns, else 1; from k = 384 an
accumulator is 2 n columns, which eligible shapes there, n <= 64, still fit twice).  So buffer 1, and the reuse of a
single buffer, only run when a CTA gets two or more tiles, i.e. from 148 * 128 + 1 rows.  MULTI_M gives every CTA 3 or
4 tiles: both buffers run at both mbarrier parities, and a single buffer is reused 3 or 4 times.

Comparison (assert_tiles): per 128-row tile, max |got - want| <= 1e-5 of that tile's own max |want|, where want is
the float64 result rounded once to fp32.  The rows of X are scaled by 2^((t mod 7) - 3) in tile t, so neighbouring
tiles of a CTA (t and t + 148) differ in scale: a tile that reads another tile's accumulator, or a stale one, is off
by far more than its own tolerance, and it cannot hide behind the scale of the other tiles.

The first two tests need no GPU: they check the C eligibility rule against a restatement of it, and that the
parametrize lists below cover the kernel's regimes."""
import math
import os

import pytest
import torch

import __graft_entry__ as entry
from deep_cbrs_amar_renaissance_b200 import _lib as L

SMS = 148                      # one persistent CTA per SM
TILE = 128                     # output rows per tile
ATOM = 32                      # fp32 columns of X per TMA load (one 128-byte swizzle row)
SLOT_BYTES = TILE * ATOM * 4   # one TMA landing slot
MAX_SLOTS = 8
SMEM = 227 * 1024              # dynamic shared memory a block may use


def landing_slots(k, n):
    """TMA landing slots that fit in shared memory beside the resident operand images of W (hi and lo halves) and the
    tail: 2 x 8 landing + 9 more mbarriers, the TMEM address word, the bias or the two attention vectors (2 n fp32)
    and 64 bytes of slack.  0: the shape does not fit with the minimum of two slots."""
    fixed = 2 * (k // ATOM) * n * 128 + (2 * MAX_SLOTS + 9) * 8 + 8 + 2 * n * 4 + 64
    if fixed + 2 * SLOT_BYTES > SMEM:
        return 0
    return min((SMEM - fixed) // SLOT_BYTES, MAX_SLOTS)


def eligible(k, n):
    return k > 0 and k % ATOM == 0 and 16 <= n <= 256 and n % 16 == 0 and landing_slots(k, n) >= 2


SPLIT_K = 384                  # from this k the cross terms Xl Wh + Xh Wl accumulate in n columns of their own


def acc_bufs(n, k):
    cols = 2 * n if k >= SPLIT_K else n
    return 2 if 2 * cols + 128 <= 512 else 1


def k_max(n):
    return max(k for k in range(ATOM, 2049, ATOM) if eligible(k, n))


WIDTHS = list(range(16, 257, 16))
MULTI_M = SMS * TILE * 3 + 77          # 445 tiles: every CTA runs 3 or 4
SMALL_MS = (1, 127, 128, 129)
ACTS = (None, "relu", "sigmoid", "tanh")
# every width at k = 32 (one atom per tile), k = 128 where it fits and the largest k (2 landing slots where n has such a
# shape): 41 shapes
SHAPES = [(n, k) for n in WIDTHS for k in sorted({ATOM, k_max(n)} | ({128} if eligible(128, n) else set()))]
# each shape at the multi-tile m and at one small m; bias + activation cycles none / relu / sigmoid / tanh over shapes
SWEEP = [(n, k, m, ACTS[i % 4]) for i, (n, k) in enumerate(SHAPES) for m in (MULTI_M, SMALL_MS[i % 4])]
EPILOGUE_WIDTHS = (16, 48, 80, 128, 192, 208, 256)


def _k_epilogue(n):
    return max(k for k in range(ATOM, 129, ATOM) if eligible(k, n))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(L.LIB_PATH):
        entry.build()
    return L.load()


# ---------------------------------------------------------------------------------------------------- no GPU needed
def test_eligibility_and_image_size_follow_the_shared_memory_rule(lib):
    for k in range(1, 2049):
        for n in range(1, 273):
            want = eligible(k, n)
            assert bool(lib.cbrs_dense_tf32x3_eligible(k, n)) == want, (k, n)
            assert lib.cbrs_dense_tf32x3_image_bytes(k, n) == (2 * (k // ATOM) * n * 128 if want else 0), (k, n)
    # anchors of the rule: the largest k per width and the landing slots left there
    assert [(n, k_max(n), landing_slots(k_max(n), n)) for n in (16, 80, 112, 128, 160, 176, 192, 208, 256)] == [
        (16, 1536, 2), (80, 288, 2), (112, 192, 3), (128, 192, 2), (160, 128, 4), (176, 128, 3), (192, 128, 2),
        (208, 96, 4), (256, 96, 2)]
    assert not any(eligible(128, n) for n in range(208, 257, 16)) and acc_bufs(192, 128) == 2 and acc_bufs(208, 96) == 1
    assert max(n for n in WIDTHS if eligible(SPLIT_K, n)) == 64 and acc_bufs(64, SPLIT_K) == 2


def test_parametrize_lists_cover_the_kernel_regimes():
    assert sorted({n for n, _ in SHAPES}) == WIDTHS
    # every CTA runs >= 3 tiles at MULTI_M, under both accumulator regimes
    assert (MULTI_M + TILE - 1) // TILE // SMS >= 3 and {acc_bufs(n, k) for n, k, m, _ in SWEEP if m == MULTI_M} == {1, 2}
    assert {k >= SPLIT_K for n, k, m, _ in SWEEP if m == MULTI_M} == {False, True}   # one and two accumulators per tile
    for n in WIDTHS:   # a 2-slot shape for each width that has one
        if any(landing_slots(k, n) == 2 for k in range(ATOM, 2049, ATOM) if eligible(k, n)):
            assert any(landing_slots(k, n) == 2 for nn, k in SHAPES if nn == n), n
    assert any(k // ATOM > landing_slots(k, n) for n, k in SHAPES)              # the landing ring wraps inside a tile
    assert {a for _, _, m, a in SWEEP if m == MULTI_M} == set(ACTS)
    assert {a for n, k, m, a in SWEEP if m == MULTI_M and acc_bufs(n, k) == 1} == set(ACTS)
    assert {acc_bufs(n, _k_epilogue(n)) for n in EPILOGUE_WIDTHS} == {1, 2}
    assert all(eligible(_k_epilogue(n), n) for n in EPILOGUE_WIDTHS)


# ---------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def dev(lib):
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _tile_scale(m, dev):
    t = torch.arange(m, device=dev) // TILE
    return torch.exp2((t % 7 - 3).to(torch.float32))[:, None]


def _inputs(m, k, n, seed, dev):
    """x [m, k] with its rows scaled per tile, w [k, n] (unit-scale products), b [n]"""
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(m, k, generator=g, device=dev) * _tile_scale(m, dev)
    w = torch.randn(k, n, generator=g, device=dev) / math.sqrt(k)
    b = torch.randn(n, generator=g, device=dev) * 0.5
    return x, w, b


ACT64 = {None: lambda v: v, "relu": lambda v: v.clamp_min(0), "sigmoid": torch.sigmoid, "tanh": torch.tanh}


def _oracle(x, w, b=None, act=None):
    v = x.double() @ w.double()
    if b is not None:
        v = v + b.double()
    return ACT64[act](v).float()


def assert_tiles(got, want, what, rtol=1e-5):
    """per 128-row tile: max |got - want| <= rtol * max |want| of that tile (NaN fails)"""
    m = want.shape[0]
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = (got.double() - want.double()).abs().reshape(m, -1).amax(1)
    mag = want.double().abs().reshape(m, -1).amax(1)
    pad = (-m) % TILE
    err = torch.nn.functional.pad(err, (0, pad)).view(-1, TILE).amax(1)
    mag = torch.nn.functional.pad(mag, (0, pad)).view(-1, TILE).amax(1)
    bad = ~(err <= rtol * mag)
    if bool(bad.any()):
        t = int(bad.nonzero()[0])
        grid = min(err.numel(), SMS)
        raise AssertionError("{}: {} of {} tiles off; first: tile {} (CTA {}, local tile {}): max err {:.3e} > {:.1e} x "
                             "{:.3e}".format(what, int(bad.sum()), err.numel(), t, t % grid, t // grid, float(err[t]), rtol,
                                             float(mag[t])))


def _image(w):
    from deep_cbrs_amar_renaissance_b200 import ops
    lib = L.load()
    k, n = w.shape
    img = torch.empty(lib.cbrs_dense_tf32x3_image_bytes(k, n), dtype=torch.uint8, device=w.device)
    L.check(lib.cbrs_dense_tf32x3_prepare(ops._ptr(w), k, n, ops._ptr(img), ops._stream()), "cbrs_dense_tf32x3_prepare")
    return img


# ---------------------------------------------------------------------------------------------------- shape sweep
@pytest.mark.gpu
@pytest.mark.parametrize("n,k,m,act", SWEEP, ids=["n%d-k%d-m%d-%s" % (n, k, m, a or "bias") for n, k, m, a in SWEEP])
def test_sweep_matches_float64_per_tile(dev, n, k, m, act):
    from deep_cbrs_amar_renaissance_b200 import ops
    x, w, b = _inputs(m, k, n, 1000 * n + k + m, dev)
    got = ops.dense_tf32x3(x, w)                                                    # kPlain
    assert_tiles(got, _oracle(x, w), "x @ w, n=%d k=%d m=%d" % (n, k, m))
    # against the FFMA kernel: within 3e-6 of the scale.  The 3xTF32 error grows linearly with k (one rounding of the
    # accumulator per MMA); at k = 1536, the deepest shape, it sits at 4.7e-6 of the scale from the FFMA result, 6e-6
    ffma = ops.dense(x, w)
    bound = 3e-6 if k <= 768 else 6e-6
    assert float((got - ffma).abs().max()) <= bound * float(ffma.abs().max())
    # bias + activation; w / 8 keeps the largest tiles' pre-activations where sigmoid and tanh are not flat
    w8 = w / 8
    got = ops.dense_tf32x3(x, w8, b, act)
    assert_tiles(got, _oracle(x, w8, b, act), "%s(x @ w + b), n=%d k=%d m=%d" % (act, n, k, m))


# ---------------------------------------------------------------------------------------------------- epilogue variants
@pytest.mark.gpu
@pytest.mark.parametrize("n", EPILOGUE_WIDTHS)
def test_bf16_output_is_the_rounded_fp32_output(dev, n):
    from deep_cbrs_amar_renaissance_b200 import ops
    k = _k_epilogue(n)
    x, w, b = _inputs(MULTI_M, k, n, 7 * n, dev)
    for args in ((), (b, "tanh")):
        full = ops.dense_tf32x3(x, w, *args)
        got = ops.dense_tf32x3(x, w, *args, out_dtype=torch.bfloat16)
        assert got.dtype == torch.bfloat16 and torch.equal(got, full.to(torch.bfloat16)), (n, k, len(args))


def _sage_oracle(x, agg, kern, b, act):
    v = torch.cat([x, agg], 1).double() @ kern.double() + b.double()
    v = v / v.pow(2).sum(1, keepdim=True).clamp_min(1e-12).sqrt()
    return ACT64[act](v).float()


@pytest.mark.gpu
@pytest.mark.parametrize("n", EPILOGUE_WIDTHS)
def test_sage_dense_runs_the_addend_l2norm_epilogue_per_tile(dev, monkeypatch, n):
    """GraphSage's dense part on the tensor cores: t = x @ K[:f], then relu(l2norm(agg @ K[f:] + t + b)) in
    cbrs_dense_tf32x3_ex; with a zero bias, the all-zero rows have a zero pre-activation (the 1e-12 clamp)"""
    from deep_cbrs_amar_renaissance_b200 import ops
    f = _k_epilogue(n)
    x, kern, b = _inputs(MULTI_M, 2 * f, n, 11 * n, dev)
    x, agg = x[:, :f].contiguous(), x[:, f:].contiguous()
    zero_rows = torch.arange(5, MULTI_M, 997, device=dev)
    x[zero_rows] = 0
    agg[zero_rows] = 0
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "tf32x3")
    for bias in (b, torch.zeros_like(b)):
        launches = ops.LAUNCHES
        got = ops.sage_dense(x, agg, kern, bias, "relu", MULTI_M)
        assert ops.LAUNCHES - launches == 4                 # the tensor-core path: two images, two products
        want = _sage_oracle(x, agg, kern, bias, "relu")
        assert_tiles(got, want, "sage dense part, n=%d f=%d" % (n, f))
        ffma = ops.dense(x, kern, bias, "relu", x2=agg, rowop=L.ROWOP_L2NORM)
        assert float((got - ffma).abs().max()) <= 3e-6
    assert not bool(got[zero_rows].any())


@pytest.mark.gpu
@pytest.mark.parametrize("n", EPILOGUE_WIDTHS)
def test_ex_entry_point_with_an_arbitrary_addend(dev, n):
    """cbrs_dense_tf32x3_ex called directly: an addend that is not a product (strided, ld_add = n + 4), rows whose
    addend is exactly -b and x = 0 (zero pre-activation), and rows whose addend cancels all of the product but a small
    residual: relu(l2norm(x @ w + addend + b)) against float64"""
    from deep_cbrs_amar_renaissance_b200 import ops
    lib = L.load()
    m, k = MULTI_M, _k_epilogue(n)
    x, w, b = _inputs(m, k, n, 13 * n, dev)
    g = torch.Generator(device=dev).manual_seed(n)
    add_buf = torch.full((m, n + 4), float("nan"), device=dev)
    addend = add_buf[:, :n]
    addend.copy_(torch.randn(m, n, generator=g, device=dev) * _tile_scale(m, dev))
    zero_rows = torch.arange(3, m, 1000, device=dev)          # rows = 3 (mod 5): none of the cancelling rows below
    x[zero_rows] = 0
    addend[zero_rows] = -b
    # near-cancelling rows in the unit-scale tiles (t mod 7 == 3): addend = -(x @ w) + a residual of 1/8 of its size
    rows = torch.arange(m, device=dev)
    cancel = rows[((rows // TILE) % 7 == 3) & (rows % 5 == 1)]
    prod = (x[cancel].double() @ w.double()).float()
    addend[cancel] = -prod + 0.125 * torch.randn(len(cancel), n, generator=g, device=dev)
    img = _image(w)
    out = torch.empty(m, n, device=dev)
    L.check(lib.cbrs_dense_tf32x3_ex(ops._ptr(x), k, ops._ptr(img), ops._ptr(b), ops._ptr(addend), n + 4,
                                     L.ROWOP_L2NORM, m, k, n, L.ACT_RELU, ops._ptr(out), n, L.DTYPE_F32, None, 0,
                                     ops._stream()), "cbrs_dense_tf32x3_ex")
    v = x.double() @ w.double() + addend.double() + b.double()
    want = (v / v.pow(2).sum(1, keepdim=True).clamp_min(1e-12).sqrt()).clamp_min(0).float()
    assert_tiles(out, want, "relu(l2norm(x @ w + addend + b)), n=%d k=%d" % (n, k))
    assert not bool(out[zero_rows].any())
    assert_tiles(out[cancel], want[cancel], "near-cancelling rows")


@pytest.mark.gpu
@pytest.mark.parametrize("n", EPILOGUE_WIDTHS)
def test_attention_logits_ride_on_the_plain_product(dev, monkeypatch, n):
    """gat_transform on the tensor cores (cbrs_dense_tf32x3_attn): z is the plain kernel's result bit for bit, and
    p = z . a_self, q = z . a_neigh are within 1e-5 of float64 per tile"""
    from deep_cbrs_amar_renaissance_b200 import ops
    k = _k_epilogue(n)
    x, w, b = _inputs(MULTI_M, k, n, 17 * n, dev)
    g = torch.Generator(device=dev).manual_seed(n + 1)
    a_s, a_n = torch.randn(n, generator=g, device=dev), torch.randn(n, generator=g, device=dev)
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "tf32x3")
    launches = ops.LAUNCHES
    z, p, q = ops.gat_transform(x, w, a_s, a_n, MULTI_M)
    assert ops.LAUNCHES - launches == 2
    assert torch.equal(z, ops.dense_tf32x3(x, w))
    z64 = x.double() @ w.double()
    assert_tiles(p, (z64 @ a_s.double()).float(), "p = z . a_self, n=%d" % n)
    assert_tiles(q, (z64 @ a_n.double()).float(), "q = z . a_neigh, n=%d" % n)


# ---------------------------------------------------------------------------------------------------- views, partitions
SENT = -7.25
G = 3   # guard rows above and below a view


@pytest.mark.gpu
@pytest.mark.parametrize("n", (80, 208))
def test_strided_views_write_nothing_outside(dev, n):
    """x read from a view inside a NaN-filled buffer; out written into views of a sentinel-filled buffer: 32-byte
    aligned rows (vector stores), 16-byte aligned rows (scalar stores), and a bf16 view"""
    from deep_cbrs_amar_renaissance_b200 import ops
    m, k = MULTI_M, _k_epilogue(n)
    x, w, b = _inputs(m, k, n, 19 * n, dev)
    xbuf = torch.full((m + 2 * G, k + 96), float("nan"), device=dev)
    xv = xbuf[G:G + m, 32:32 + k]
    xv.copy_(x)
    for args in ((), (b, "sigmoid")):
        full = ops.dense_tf32x3(x, w, *args)
        for col, extra, dtype in ((8, 40, torch.float32), (4, 36, torch.float32), (16, 48, torch.bfloat16)):
            obuf = torch.full((m + 2 * G, n + extra), SENT, device=dev, dtype=dtype)
            ov = obuf[G:G + m, col:col + n]
            ops.dense_tf32x3(xv, w, *args, out=ov)
            assert torch.equal(ov, full.to(dtype)), (n, col, dtype)
            ov.fill_(SENT)
            assert bool((obuf == SENT).all()), "wrote outside the view (n=%d, column %d, %s)" % (n, col, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("n", (80, 208))
def test_row_slices_are_bit_equal_to_the_full_run(dev, monkeypatch, n):
    """row partitions start anywhere in a tile and span more than one wave of CTAs: same bits as the full run, for
    the plain, bias + activation, attention and addend + l2norm epilogues"""
    from deep_cbrs_amar_renaissance_b200 import ops
    m, k = MULTI_M, _k_epilogue(n)
    x, w, b = _inputs(m, k, n, 23 * n, dev)
    agg = torch.flip(x, (0,)).contiguous()
    kern = torch.cat([w, torch.flip(w, (0,))]).contiguous()
    a_s, a_n = b, torch.flip(b, (0,)).contiguous()
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "tf32x3")
    runs = {
        "plain": lambda a, e: ops.dense_tf32x3(x[a:e], w),
        "bias+tanh": lambda a, e: ops.dense_tf32x3(x[a:e], w, b, "tanh"),
        "attn": lambda a, e: torch.cat([z.reshape(e - a, -1) for z in ops.gat_transform(x[a:e], w, a_s, a_n, m)], 1),
        "sage": lambda a, e: ops.sage_dense(x[a:e], agg[a:e], kern, b, "relu", m),
    }
    wave = SMS * TILE
    for name, run in runs.items():
        full = run(0, m)
        for a, e in ((37, 37 + wave + 500), (200, m), (m - wave - 129, m - 1), (64, 2 * wave + 64)):
            assert torch.equal(run(a, e), full[a:e]), (name, n, a, e)


# ---------------------------------------------------------------------------------------------------- dispatch
# (k, n, what gat_transform does when the tensor-core kernel refuses the shape: the FFMA kernel's attention row-op
# takes n <= 128 only)
DISPATCH = [(128, 128, None), (32, 16, None), (1536, 16, None), (192, 128, None), (96, 208, None), (96, 256, None),
            (128, 192, None), (160, 144, None),
            (128, 208, "raises"), (128, 256, "raises"), (192, 144, "raises"), (1568, 16, "ffma"), (224, 128, "ffma"),
            (40, 64, "ffma"), (64, 24, "ffma"), (64, 272, "raises")]


@pytest.mark.gpu
@pytest.mark.parametrize("k,n,gat_refused", DISPATCH, ids=["k%d-n%d" % (k, n) for k, n, _ in DISPATCH])
def test_dispatch_follows_the_c_predicate(dev, monkeypatch, k, n, gat_refused):
    """gcn_transform, sage_dense and gat_transform take the tensor-core kernel exactly when tf32x3_chosen says so, and
    that is the C predicate from TF32X3_MIN_ROWS graph nodes up.  Where the kernel refuses the shape, gcn_transform
    and sage_dense return the FFMA kernel's float64-accurate result; gat_transform does too for n <= 128 and raises
    CbrsError above"""
    from deep_cbrs_amar_renaissance_b200 import ops
    ok = eligible(k, n)
    assert (gat_refused is None) == ok
    big = ops.TF32X3_MIN_ROWS
    assert ops.tf32x3_chosen(big, k, n) == ok and not ops.tf32x3_chosen(big - 1, k, n)
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "ffma")
    assert not ops.tf32x3_chosen(big, k, n)
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "tf32x3")
    assert ops.tf32x3_chosen(1, k, n) == ok
    monkeypatch.setattr(ops, "GCN_TRANSFORM", "auto")

    m = 300
    x, w, b = _inputs(m, k, n, k + n, dev)
    agg = torch.flip(x, (0,)).contiguous()
    kern = torch.cat([w, w.flip(0)]).contiguous()
    a_s, a_n = b, b.flip(0).contiguous()
    want = _oracle(x, w)

    z = ops.gcn_transform(x, w, big)
    assert torch.equal(z, ops.dense_tf32x3(x, w) if ok else ops.dense(x, w))
    assert_tiles(z, want, "gcn_transform k=%d n=%d" % (k, n))
    assert torch.equal(ops.gcn_transform(x, w, big - 1), ops.dense(x, w))

    launches = ops.LAUNCHES
    s = ops.sage_dense(x, agg, kern, b, "relu", big)
    assert ops.LAUNCHES - launches == (4 if ok else 1 + (n > 128))
    if not ok:
        assert torch.equal(s, ops.dense(x, kern, b, "relu", x2=agg, rowop=L.ROWOP_L2NORM))
    assert_tiles(s, _sage_oracle(x, agg, kern, b, "relu"), "sage_dense k=%d n=%d" % (k, n))

    if gat_refused == "raises":
        with pytest.raises(L.CbrsError, match="n <= 128"):
            ops.gat_transform(x, w, a_s, a_n, big)
        return
    zz, p, q = ops.gat_transform(x, w, a_s, a_n, big)
    if ok:
        assert torch.equal(zz, ops.dense_tf32x3(x, w))
    else:
        zf, pf, qf = ops.dense(x, w, rowop=L.ROWOP_ATTN, a_self=a_s, a_neigh=a_n)
        assert torch.equal(zz, zf) and torch.equal(p, pf) and torch.equal(q, qf)
    z64 = x.double() @ w.double()
    assert_tiles(zz, want, "gat_transform z")
    assert_tiles(p, (z64 @ a_s.double()).float(), "gat_transform p")
    assert_tiles(q, (z64 @ a_n.double()).float(), "gat_transform q")


@pytest.mark.gpu
@pytest.mark.parametrize("k,n", ((128, 128), (96, 208)))
def test_dispatch_follows_the_alignment_rules(dev, k, n):
    """an eligible shape still goes to the FFMA kernel when x or out breaks the TMA / vector-store alignment: rows of x
    not a multiple of 16 bytes apart or not 16-byte aligned, fp32 out rows not 16-byte aligned, bf16 out rows not
    32-byte aligned; aligned strided views take the tensor cores"""
    from deep_cbrs_amar_renaissance_b200 import ops
    m = 300
    big = ops.TF32X3_MIN_ROWS
    x, w, _ = _inputs(m, k, n, 5 * k + n, dev)
    want = _oracle(x, w)
    tc, ffma = ops.dense_tf32x3(x, w), ops.dense(x, w)
    xs = {"aligned view": (torch.zeros(m, k + 32, device=dev)[:, 32:], True),
          "ldx % 4 != 0": (torch.zeros(m, k + 2, device=dev)[:, :k], False),
          "x + 4 bytes": (torch.zeros(m, k + 4, device=dev)[:, 1:1 + k], False)}
    for name, (xv, ok) in xs.items():
        xv.copy_(x)
        assert ops.tf32x3_chosen(big, k, n, xv) == ok, name
        z = ops.gcn_transform(xv, w, big)
        assert torch.equal(z, tc if ok else ops.dense(xv, w)), name   # the FFMA kernel's variant depends on x's alignment
        assert_tiles(z, want, name)
    outs = {"fp32 aligned view": (torch.float32, 8, 16, True), "fp32 + 8 bytes": (torch.float32, 2, 16, False),
            "fp32 ldo % 4 != 0": (torch.float32, 0, 2, False), "bf16 aligned view": (torch.bfloat16, 16, 32, True),
            "bf16 + 16 bytes": (torch.bfloat16, 8, 32, False), "bf16 ldo % 16 != 0": (torch.bfloat16, 0, 8, False)}
    for name, (dtype, col, extra, ok) in outs.items():
        buf = torch.full((m, n + extra), SENT, device=dev, dtype=dtype)
        ov = buf[:, col:col + n]
        assert ops.tf32x3_chosen(big, k, n, x, ov) == ok, name
        assert ops.gcn_transform(x, w, big, out=ov) is ov
        assert torch.equal(ov, (tc if ok else ffma).to(dtype)), name
        ov.fill_(SENT)
        assert bool((buf == SENT).all()), name
