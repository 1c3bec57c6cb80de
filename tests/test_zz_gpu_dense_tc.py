"""cbrs_dense_tc: the Dense layer on the tensor cores (tcgen05, bf16 operands, fp32 accumulate) against an oracle that
rounds the same operands to bf16 and sums in float64.  Tolerance 1e-4 of the output scale pre-activation-wise (fp32
accumulation order inside the tensor core is not specified; a layout or descriptor bug gives O(1) errors).
Model level: a hybrid model with set_scorer_precision('bf16') against the same rounding oracle, and against its own
fp32 scores within 2e-2."""
import numpy as np
import pytest
import torch

from oracle import layers as ol

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _device():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)


def oracle_dense_bf16(a, w, b, act):
    y = ol.bf16_round(a).astype(np.float64) @ ol.bf16_round(w).astype(np.float64)
    if b is not None:
        y = y + b.astype(np.float64)
    return ol.activation(act)(y.astype(np.float32))


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def close(got, want, what, rtol=1e-4):
    scale = max(np.abs(want).max(), 1e-30)
    err = np.abs(got.astype(np.float64) - want.astype(np.float64)).max()
    assert err <= rtol * scale, "{}: max abs err {:.3e} (scale {:.3e})".format(what, err, scale)


# k < 512 runs dense_tc_kernel, k >= 512 dense_tc_x_kernel: each kernel at the same widths, activations and bias settings
@pytest.mark.parametrize("m,k,n,act,bias", [(300, 768, 256, "relu", True), (128, 64, 64, None, True), (77, 24, 16, "tanh", False),
                                            (1000, 200, 40, None, True), (5, 256, 8, "sigmoid", True), (4097, 128, 128, "relu", True),
                                            (128, 576, 64, None, True), (77, 512, 16, "tanh", False), (1000, 520, 40, None, True),
                                            (5, 768, 8, "sigmoid", True), (4097, 1024, 128, "relu", True)])
def test_dense_tc_single_source(m, k, n, act, bias):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(m + k + n)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (rng.standard_normal((k, n)) / np.sqrt(k)).astype(np.float32)
    b = (rng.standard_normal(n) * 0.1).astype(np.float32) if bias else None
    got = ops.dense_tc(cuda(a), cuda(w), cuda(b) if bias else None, act).cpu().numpy()
    assert got.shape == (m, n)
    close(got, oracle_dense_bf16(a, w, b, act), "dense_tc %dx%dx%d %s" % (m, k, n, act))


def _gather_concat_strided(f1, f2, n, seed):
    """two gathered sources (the scorer's lookup + concat), a column-slice source and a strided output"""
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(seed)
    t1 = rng.standard_normal((500, f1 + 8)).astype(np.float32)
    t2 = rng.standard_normal((400, f2)).astype(np.float32)
    i1 = rng.randint(0, 500, size=1000)
    i1[:64] = i1[0]
    i2 = rng.randint(0, 400, size=1000)
    w = (rng.standard_normal((f1 + f2, n)) / np.sqrt(f1 + f2)).astype(np.float32)
    b = (rng.standard_normal(n) * 0.1).astype(np.float32)
    src1 = cuda(t1)[:, 4:4 + f1]        # ld f1 + 8, offset 16 bytes
    buf = torch.zeros(1000, n + 8, device="cuda")
    out = ops.dense_tc(src1, cuda(w), cuda(b), "sigmoid", x2=cuda(t2), idx1=cuda(i1), idx2=cuda(i2), out=buf[:, 4:4 + n])
    a = np.concatenate([t1[i1][:, 4:4 + f1], t2[i2]], axis=1)
    close(out.cpu().numpy(), oracle_dense_bf16(a, w, b, "sigmoid"), "gather + concat %d + %d -> %d" % (f1, f2, n))
    assert float(buf[:, :4].abs().max()) == 0.0 and float(buf[:, 4 + n:].abs().max()) == 0.0   # nothing written outside the view
    # a prepared image can be reused across calls
    image = ops.dense_tc_image(cuda(w))
    again = ops.dense_tc(src1, cuda(w), cuda(b), "sigmoid", x2=cuda(t2), idx1=cuda(i1), idx2=cuda(i2), image=image)
    assert torch.equal(again, out.contiguous())


def test_dense_tc_gather_concat_strided():
    _gather_concat_strided(96, 48, 64, seed=1)


def test_dense_tc_gather_concat_strided_deep():
    """the same at the depth of the hybrid scorer's concatenated towers (f1 + f2 >= 512: dense_tc_x_kernel)"""
    _gather_concat_strided(512, 256, 64, seed=2)


@pytest.mark.parametrize("f1,f2,kernel", [(504, 0, "dense_tc_kernel"), (512, 0, "dense_tc_x_kernel"),
                                          (256, 248, "dense_tc_kernel"), (256, 256, "dense_tc_x_kernel")])
def test_dense_tc_kernel_chosen_by_depth(f1, f2, kernel):
    """cbrs_dense_tc runs dense_tc_x_kernel from f1 + f2 = 512 up and dense_tc_kernel below, whatever the split"""
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(f1 + f2)
    m, n = 300, 64
    a = rng.standard_normal((m, f1 + f2)).astype(np.float32)
    w = (rng.standard_normal((f1 + f2, n)) / np.sqrt(f1 + f2)).astype(np.float32)
    b = (rng.standard_normal(n) * 0.1).astype(np.float32)
    x1, x2 = cuda(a[:, :f1]), (cuda(a[:, f1:]) if f2 else None)
    wd, bd = cuda(w), cuda(b)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        got = ops.dense_tc(x1, wd, bd, "relu", x2=x2)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    ran = {k for k in ("dense_tc_kernel", "dense_tc_x_kernel") if any(k in name for name in names)}
    assert ran == {kernel}, sorted(name for name in names if "dense_tc" in name)
    close(got.cpu().numpy(), oracle_dense_bf16(a, w, b, "relu"), "dense_tc %d + %d -> %d" % (f1, f2, n))


def test_dense_tc_refuses_what_it_cannot_take():
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    x = torch.zeros(16, 20, device="cuda")
    with pytest.raises(_lib.CbrsError, match="multiples of 8"):
        ops.dense_tc(x, torch.zeros(20, 16, device="cuda"))
    with pytest.raises(_lib.CbrsError, match="n <= 256"):
        ops.dense_tc(torch.zeros(16, 64, device="cuda"), torch.zeros(64, 512, device="cuda"))
    assert not ops.dense_tc_eligible(20, 0, 16) and not ops.dense_tc_eligible(64, 0, 512) and ops.dense_tc_eligible(768, 0, 256)


def test_hybrid_scorer_on_tensor_cores():
    """HybridBertGCN at the grid-2 shapes of econfigs/hybrid-gnn.yaml (BERT towers 768 -> 256 -> 64): bf16 scorer vs the
    rounding oracle layer by layer, and vs the fp32 scorer"""
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import hybrid
    from tests.helpers import export_weights, random_bipartite
    from tests.test_gpu_models import _randomise
    set_seed(42)
    n_users, n_items, b = 300, 200, 2048
    adj = random_bipartite(n_users, n_items, 6000, seed=7)
    model = hybrid.HybridBertGCN(adj, embedding_dim=16, n_hiddens=[16, 16], dense_units=[[48, 48], [256, 64], [64, 64]],
                                 clf_units=[64, 64], feature_based=True, l2_regularizer=1e-4)
    rng = np.random.RandomState(3)
    table = (rng.standard_normal((n_users + n_items, 768)) * 0.5).astype(np.float32)
    u = rng.randint(0, n_users, size=b)
    i = rng.randint(0, n_items, size=b) + n_users
    model.set_content_table(table)
    fp32 = model((u, i)).cpu().numpy()
    _randomise(model, seed=4)
    fp32 = model((u, i)).cpu().numpy()
    launches = ops.LAUNCHES
    model.set_scorer_precision("bf16")
    got = model((u, i)).cpu().numpy()
    assert ops.LAUNCHES > launches
    model.set_scorer_precision("fp32")
    assert np.array_equal(model((u, i)).cpu().numpy(), fp32)
    assert np.abs(got - fp32).max() <= 2e-2
    # the rounding oracle: every Dense rounds its input and its kernel to bf16 (widths 48, 768, 256, 96, 128, 64 are
    # all multiples of 8 and <= 256 outputs, so every layer of this scorer takes the tensor-core kernel)
    w = export_weights(model)
    emb = model.gnn(None).cpu().numpy()

    def stack(x, layers, last=None):
        for k, (kern, bias) in enumerate(layers):
            x = oracle_dense_bf16(x, kern, bias, last if (last and k == len(layers) - 1) else "relu")
        return x

    ug, ig = stack(emb[u], w["dense1a"]), stack(emb[i], w["dense1b"])
    ub, ib = stack(table[u], w["dense2a"]), stack(table[i], w["dense2b"])
    x1 = stack(np.concatenate([ug, ig], 1), w["dense3a"])
    x2 = stack(np.concatenate([ub, ib], 1), w["dense3b"])
    want = stack(np.concatenate([x1, x2], 1), w["clf"], last="sigmoid")
    close(got, want, "bf16 hybrid scores", rtol=2e-3)   # bf16 re-rounding of near-tie activations between layers
