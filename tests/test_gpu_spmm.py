# coding=utf-8
"""GPU parity for K1 (tfgk_spmm_f32) through the reference-facing API.
SUM / MEAN are BIT-EXACT against the oracle (same sequential fp32 order as tf.math.unsorted_segment_sum on CPU),
MAX is exact by construction."""
import numpy as np
import pytest
import torch

import tf_geometric_b200 as tfg
from tf_geometric_b200 import ops
from oracle import tfg_oracle as o
from oracle import c_oracle
from conftest import random_graph, assert_close

pytestmark = pytest.mark.gpu


def dev(a, dtype=None):
    return ops.as_device(a, dtype)


def host(t):
    return t.detach().cpu().numpy()


GRAPH = dict(n=3000, e=45000, seed=5, isolated=11, hub=(42, 1900))     # <= ops.HUB_THRESHOLD: strictly sequential rows


def _graph():
    ei = random_graph(GRAPH["n"], GRAPH["e"], GRAPH["seed"], isolated=GRAPH["isolated"], hub=GRAPH["hub"])
    return ei, GRAPH["n"]


@pytest.mark.parametrize("d", [1, 2, 3, 4, 7, 8, 16, 20, 33, 64, 100, 128, 130, 256, 300, 384, 512, 516, 1000])
@pytest.mark.parametrize("weighted", [False, True])
def test_aggregate_sum_bit_exact_all_widths(d, weighted):
    ei, n = _graph()
    rs = np.random.RandomState(d)
    x = rs.randn(n, d).astype(np.float32)
    w = rs.rand(ei.shape[1]).astype(np.float32) if weighted else None
    want = c_oracle.aggregate(ei[0], ei[1], w, x, n, "sum")
    got = tfg.nn.aggregate_neighbors(dev(x), dev(ei), dev(w), mapper=tfg.nn.gcn_mapper if weighted else tfg.nn.identity_mapper,
                                     reducer=tfg.nn.sum_reducer, updater=tfg.nn.identity_updater)
    np.testing.assert_array_equal(host(got), want)


@pytest.mark.parametrize("d", [1, 7, 16, 100, 128, 200])
@pytest.mark.parametrize("reduce", ["mean", "max"])
def test_aggregate_mean_max(d, reduce):
    ei, n = _graph()
    rs = np.random.RandomState(d + 1)
    x = rs.randn(n, d).astype(np.float32)
    w = rs.rand(ei.shape[1]).astype(np.float32)
    reducer = {"mean": tfg.nn.mean_reducer, "max": tfg.nn.max_reducer}[reduce]
    for weights, mapper in ((None, tfg.nn.identity_mapper), (w, tfg.nn.gcn_mapper)):
        want = c_oracle.aggregate(ei[0], ei[1], weights, x, n, reduce)
        got = tfg.nn.aggregate_neighbors(dev(x), dev(ei), dev(weights), mapper=mapper, reducer=reducer,
                                         updater=tfg.nn.identity_updater)
        np.testing.assert_array_equal(host(got), want)
    # empty segments: mean -> 0, max -> float32 lowest (TF2 unsorted_segment_max)
    got = host(got)
    assert (got[:GRAPH["isolated"]] == (0.0 if reduce == "mean" else np.finfo(np.float32).min)).all()


def test_aggregate_defaults_sum_updater_and_empty_edge_index():
    ei, n = _graph()
    x = np.random.RandomState(0).randn(n, 24).astype(np.float32)
    want = o.aggregate_neighbors(x, ei)                       # identity_mapper, sum_reducer, sum_updater
    got = tfg.nn.aggregate_neighbors(dev(x), dev(ei))
    np.testing.assert_array_equal(host(got), want)
    xd = dev(x)
    assert tfg.nn.aggregate_neighbors(xd, []) is xd            # map_reduce.py:57-58


def test_generic_mapper_route_and_standalone_reducers():
    ei, n = _graph()
    rs = np.random.RandomState(3)
    x = rs.randn(n, 12).astype(np.float32)

    def my_mapper(repeated_x, neighbor_x, edge_weight=None):
        return neighbor_x - repeated_x

    want = o.aggregate_neighbors(x, ei, mapper=lambda r, nb, edge_weight=None: nb - r, reducer=o.mean_reducer,
                                 updater=o.identity_updater)
    got = tfg.nn.aggregate_neighbors(dev(x), dev(ei), mapper=my_mapper, reducer=tfg.nn.mean_reducer,
                                     updater=tfg.nn.identity_updater)
    np.testing.assert_array_equal(host(got), want)
    msg = rs.randn(ei.shape[1], 5).astype(np.float32)
    for fn_g, fn_o in ((tfg.nn.sum_reducer, o.sum_reducer), (tfg.nn.mean_reducer, o.mean_reducer),
                       (tfg.nn.max_reducer, o.max_reducer)):
        np.testing.assert_array_equal(host(fn_g(dev(msg), dev(ei[0]), num_nodes=n)), fn_o(msg, ei[0], n))
    cnt = tfg.nn.aggregate_neighbors(dev(x), dev(ei), mapper=tfg.nn.neighbor_count_mapper, reducer=tfg.nn.sum_reducer,
                                     updater=tfg.nn.identity_updater)
    np.testing.assert_array_equal(host(cnt)[:, 0], np.bincount(ei[0], minlength=n).astype(np.float32))


def test_spmm_epilogue_bias_relu_axpby_strided():
    ei, n = _graph()
    rs = np.random.RandomState(9)
    d = 40
    big = rs.randn(n, 3 * d).astype(np.float32)
    h = dev(big)[:, d:2 * d]                                   # strided view: ldh = 3d
    w = rs.rand(ei.shape[1]).astype(np.float32)
    bias = rs.randn(d).astype(np.float32)
    add = rs.randn(n, d).astype(np.float32)
    adj = tfg.SparseMatrix(ei, w, [n, n])
    agg = c_oracle.aggregate(ei[0], ei[1], w, big[:, d:2 * d], n, "sum")
    got = adj.matmul(h, bias=dev(bias), act=ops.ACT_RELU)
    np.testing.assert_array_equal(host(got), np.maximum(agg + bias, 0))
    got = adj.matmul(h, alpha=0.9, addend=dev(add), beta=0.1)
    np.testing.assert_array_equal(host(got), (agg * np.float32(0.9) + add * np.float32(0.1)).astype(np.float32))
    out = torch.zeros((n, 2 * d), dtype=torch.float32, device="cuda")
    adj.matmul(h, out=out[:, d:])
    np.testing.assert_array_equal(host(out[:, d:]), agg)
    assert (host(out[:, :d]) == 0).all()


def test_spmm_matches_dense_float64_model():
    ei, n = _graph()
    rs = np.random.RandomState(11)
    w = rs.rand(ei.shape[1]).astype(np.float32)
    h = rs.randn(n, 16).astype(np.float32)
    got = tfg.SparseMatrix(ei, w, [n, n]) @ dev(h)
    assert_close(host(got), o.dense_spmm_f64(ei, w, [n, n], h), rtol=1e-4, atol_scale=1e-6, what="spmm vs dense f64")


def test_determinism_run_to_run():
    ei, n = _graph()
    rs = np.random.RandomState(13)
    x = dev(rs.randn(n, 128).astype(np.float32))
    adj = tfg.SparseMatrix(ei, rs.rand(ei.shape[1]).astype(np.float32), [n, n])
    first = host(adj @ x)
    for _ in range(3):
        np.testing.assert_array_equal(host(adj @ x), first)


@pytest.mark.parametrize("d", [128, 100, 32, 200])
def test_hub_rows_are_sliced_and_merged_deterministically(d):
    """Rows above ops.HUB_THRESHOLD edges are reduced in 2048-edge slices by separate warps and merged in slice order:
    every other row stays bit-identical to the sequential oracle, hub rows agree to fp32 rounding, runs are repeatable."""
    n = 20000
    rs = np.random.RandomState(d)
    base = random_graph(n, 150000, seed=3, isolated=3)
    hubs = {7: 5000, 123: 70000, 19999: 2049, 4000: 1500}          # 4000 stays below the threshold (with its base edges)
    extra = [np.stack([np.full(k, node), rs.randint(0, n, k)]) for node, k in hubs.items()]
    ei = np.concatenate([base] + extra, axis=1).astype(np.int32)
    ei = ei[:, rs.permutation(ei.shape[1])]
    w = rs.rand(ei.shape[1]).astype(np.float32)
    x = rs.randn(n, d).astype(np.float32)
    csr = ops.csr_build(dev(ei[0]), dev(ei[1]), n)
    deg = np.bincount(ei[0], minlength=n)
    is_hub = deg > ops.HUB_THRESHOLD
    assert csr.plan is not None and csr.plan.n_hubs == int(is_hub.sum()) and is_hub[[7, 123, 19999]].all() and not is_hub[4000]
    assert deg[4000] <= ops.HUB_THRESHOLD
    assert csr.plan.n_slots == int(np.ceil(deg[is_hub] / ops.HUB_CHUNK).sum())
    w_csr = ops.permute(dev(w), csr.perm)
    for reduce in ("sum", "mean", "max"):
        want = c_oracle.aggregate(ei[0], ei[1], w, x, n, reduce)
        got = host(ops.spmm(csr, w_csr, dev(x), reduce=reduce))
        np.testing.assert_array_equal(got[~is_hub], want[~is_hub])
        if reduce == "max":
            np.testing.assert_array_equal(got[is_hub], want[is_hub])
        else:
            scale = np.abs(want[is_hub]).max()
            assert np.abs(got[is_hub] - want[is_hub]).max() <= 2e-5 * scale
        np.testing.assert_array_equal(host(ops.spmm(csr, w_csr, dev(x), reduce=reduce)), got)
    bias = rs.randn(d).astype(np.float32)
    add = rs.randn(n, d).astype(np.float32)
    want = np.maximum(c_oracle.aggregate(ei[0], ei[1], w, x, n, "sum") * np.float32(0.5) + add * np.float32(2.0) + bias, 0)
    got = host(ops.spmm(csr, w_csr, dev(x), alpha=0.5, addend=dev(add), beta=2.0, bias=dev(bias), act=ops.ACT_RELU))
    np.testing.assert_array_equal(got[~is_hub], want[~is_hub])
    assert np.abs(got[is_hub] - want[is_hub]).max() <= 2e-5 * np.abs(want).max()


@pytest.mark.parametrize("d", [128, 100, 64, 32, 256, 200])
@pytest.mark.parametrize("reduce", ["sum", "mean", "max"])
def test_tma_gather4_variant_is_bit_identical(d, reduce):
    """K1 through TMA tile::gather4 (one instruction fetches four neighbour rows into the warp's ring), the kernel for float4
    rows of 32..256 columns: bias + ReLU epilogue, ragged rows, empty rows and a hub row cut into slices.  Every row but the
    hub is bit-identical to the sequential oracle, the hub row agrees to fp32 rounding, and runs are repeatable."""
    rs = np.random.RandomState(d)
    n = 3000
    ei = random_graph(n, 40000, seed=d, isolated=7, hub=(11, 9000))
    csr = ops.csr_build(dev(ei[0]), dev(ei[1]), n, n)
    deg = np.bincount(ei[0], minlength=n)
    is_hub = deg > ops.HUB_THRESHOLD
    assert csr.plan is not None and csr.plan.n_hubs == int(is_hub.sum()) and is_hub[11]
    w = (rs.rand(ei.shape[1]) + 0.1).astype(np.float32) if reduce != "mean" else None
    w_csr = ops.permute(dev(w), csr.perm) if w is not None else None
    x = rs.randn(n, d).astype(np.float32)
    bias = rs.randn(d).astype(np.float32)
    want = np.maximum(c_oracle.aggregate(ei[0], ei[1], w, x, n, reduce) + bias, 0)
    got = ops.spmm(csr, w_csr, dev(x), reduce=reduce, bias=dev(bias), act=ops.ACT_RELU)
    out = host(got)
    np.testing.assert_array_equal(out[~is_hub], want[~is_hub])
    assert np.abs(out[is_hub] - want[is_hub]).max() <= 2e-5 * np.abs(want[is_hub]).max()
    again = ops.spmm(csr, w_csr, dev(x), reduce=reduce, bias=dev(bias), act=ops.ACT_RELU)
    assert torch.equal(again, got), "gather4 is not repeatable (D={}, reduce={})".format(d, reduce)
