# coding=utf-8
"""GPU parity for K3: segment_softmax and the fused GAT kernel (fast float4 path and generic path)."""
import numpy as np
import pytest
import torch

import tf_geometric_b200 as tfg
from tf_geometric_b200 import ops
from oracle import tfg_oracle as o
from oracle import c_oracle
from conftest import random_graph, assert_close, glorot

pytestmark = pytest.mark.gpu


def dev(a, dtype=None):
    return ops.as_device(a, dtype)


def host(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("cols", [None, 1, 3, 8])
def test_segment_softmax(cols):
    rs = np.random.RandomState(0)
    n, e = 500, 12000
    ids = np.concatenate([rs.randint(5, n, e), np.full(3000, 7)]).astype(np.int32)    # segment 7 is a hub, 0..4 empty
    rs.shuffle(ids)
    data = (rs.randn(len(ids)) * 4).astype(np.float32) if cols is None else (rs.randn(len(ids), cols) * 4).astype(np.float32)
    got = host(tfg.nn.segment_softmax(dev(data), dev(ids), n))
    if cols is None:
        want = o.segment_softmax(data, ids, n)
    else:
        want = np.stack([o.segment_softmax(data[:, i], ids, n) for i in range(cols)], axis=1)
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-9)
    sums = np.zeros((n,) + got.shape[1:], np.float64)
    np.add.at(sums, ids, got.astype(np.float64))
    np.testing.assert_allclose(sums[np.unique(ids)], 1.0, atol=1e-5)


CASES = [
    # f, attention_units, units, heads, split, isolated/hub graph
    (24, 128, 128, 8, True),     # cfg3 shape: head dim 16 (fast path, NCK=NCV=1)
    (24, 64, 64, 8, True),       # demo-like, head dim 8
    (24, 32, 16, 8, True),       # dqk 4, dv 2 (dv % 4 != 0 -> generic)
    (10, 8, 64, 8, True),        # demo_gat.py: attention_units=8, 8 heads -> dqk = 1 (generic)
    (16, 256, 256, 4, True),     # NCK = NCV = 2
    (16, 512, 384, 8, True),     # NCK = 4, NCV = 3
    (16, 96, 96, 8, True),       # dqk = 12 -> 3 lanes per head (not a power of two -> generic)
    (16, 48, 40, 4, False),      # averaged heads (generic), V is [N, units * heads]
    (16, 16, 12, 1, True),       # single head
    (16, 128, 128, 32, True),    # 32 heads, dqk = 4
]


@pytest.mark.parametrize("f,a,u,heads,split", CASES)
def test_gat_forward_matches_oracle(f, a, u, heads, split):
    rs = np.random.RandomState(a + u + heads)
    n = 1200
    ei = random_graph(n, 14000, seed=heads, isolated=3, hub=(9, 1500))
    ei = np.concatenate([ei, np.array([[5, 5], [5, 5]], np.int32)], axis=1)    # pre-existing self loop, twice
    x = rs.randn(n, f).astype(np.float32)
    wq, wk = glorot(rs, f, a), glorot(rs, f, a)
    wv = glorot(rs, f, u if split else u * heads)
    bq, bk = (rs.randn(a) * .1).astype(np.float32), (rs.randn(a) * .1).astype(np.float32)
    b = rs.randn(u).astype(np.float32)
    want, want_att = o.gat(x, ei, wq, bq, o.relu, wk, bk, o.relu, wv, b, o.relu, num_heads=heads,
                           split_value_heads=split, return_attention=True)
    got, got_att = tfg.nn.gat(dev(x), dev(ei), dev(wq), dev(bq), tfg.nn.relu, dev(wk), dev(bk), tfg.nn.relu, dev(wv),
                              dev(b), tfg.nn.relu, num_heads=heads, split_value_heads=split, return_attention=True)
    assert_close(host(got), want, what="gat out")
    np.testing.assert_allclose(host(got_att), want_att, rtol=1e-4, atol=1e-7)
    again = tfg.nn.gat(dev(x), dev(ei), dev(wq), dev(bq), tfg.nn.relu, dev(wk), dev(bk), tfg.nn.relu, dev(wv),
                       dev(b), tfg.nn.relu, num_heads=heads, split_value_heads=split)
    assert_close(host(again), host(got), rtol=1e-5, atol_scale=1e-6, what="gat with/without attention output")
    once_more = tfg.nn.gat(dev(x), dev(ei), dev(wq), dev(bq), tfg.nn.relu, dev(wk), dev(bk), tfg.nn.relu, dev(wv),
                           dev(b), tfg.nn.relu, num_heads=heads, split_value_heads=split)
    np.testing.assert_array_equal(host(once_more), host(again))     # the same call is bit-for-bit deterministic


def test_gat_kernel_core_tight_against_c_oracle():
    """Same Q/K/V handed to both sides: isolates the fused kernel from the dense projections (tolerance 2e-6 rel)."""
    rs = np.random.RandomState(1)
    n, heads, a, u = 4000, 8, 128, 128
    ei = random_graph(n, 90000, seed=3, hub=(100, 5000))
    full, _ = o.add_self_loop_edge(ei, n)
    q, k, v = (rs.randn(n, d).astype(np.float32) for d in (a, a, u))
    want, want_att = c_oracle.gat_core(full[0], full[1], q, k, v, heads, True, return_attention=True)
    csr = ops.csr_build(dev(full[0]), dev(full[1]), n)
    got, att = ops.gat_fused(csr, dev(q), dev(k), dev(v), heads, return_attention=True)
    assert_close(host(got), want, rtol=2e-5, atol_scale=2e-6, what="gat core")
    np.testing.assert_allclose(host(att), want_att[host(csr.perm)], rtol=2e-5, atol=1e-9)


def test_gat_layer_defaults_and_weight_names():
    rs = np.random.RandomState(2)
    n, f = 300, 20
    ei = random_graph(n, 2500, seed=6)
    x = rs.randn(n, f).astype(np.float32)
    layer = tfg.layers.GAT(64, num_heads=8, attention_units=8, activation=tfg.nn.relu, seed=1)     # demo_gat.py:21
    out = layer([dev(x), dev(ei)])
    names = sorted(k for k, _ in layer.named_parameters())
    assert names == ["bias", "kernel", "key_bias", "key_kernel", "query_bias", "query_kernel"]
    p = {k: host(v) for k, v in layer.named_parameters()}
    assert p["query_kernel"].shape == (f, 8) and p["kernel"].shape == (f, 64) and (p["bias"] == 0).all()
    want = o.gat(x, ei, p["query_kernel"], p["query_bias"], o.relu, p["key_kernel"], p["key_bias"], o.relu,
                 p["kernel"], p["bias"], o.relu, num_heads=8)
    assert_close(host(out), want, what="GAT layer")


def test_gat_hub_rows_sliced_softmax_merge():
    """Hub rows in the fused GAT: per-slice (sum, max, denominator) partials merged with the log-sum-exp rule."""
    rs = np.random.RandomState(5)
    n, heads, a = 30000, 8, 128
    base = random_graph(n, 200000, seed=9)
    extra = [np.stack([np.full(k, node), rs.randint(0, n, k)]) for node, k in ((11, 9000), (29999, 120000), (500, 2100))]
    ei = np.concatenate([base] + extra, axis=1).astype(np.int32)
    ei = ei[:, rs.permutation(ei.shape[1])]
    full, _ = o.add_self_loop_edge(ei, n)
    q, k, v = (rs.randn(n, a).astype(np.float32) for _ in range(3))
    want = c_oracle.gat_core(full[0], full[1], q, k, v, heads, True)
    csr = ops.csr_build(dev(full[0]), dev(full[1]), n)
    assert csr.plan is not None and csr.plan.n_hubs == 3
    got = ops.gat_fused(csr, dev(q), dev(k), dev(v), heads)
    assert_close(host(got), want, rtol=2e-5, atol_scale=2e-6, what="gat with hub rows")
    assert torch.equal(got, ops.gat_fused(csr, dev(q), dev(k), dev(v), heads))
    got_att, att = ops.gat_fused(csr, dev(q), dev(k), dev(v), heads, return_attention=True)   # per-row kernel, same answer
    assert_close(host(got_att), want, rtol=2e-5, atol_scale=2e-6, what="gat with hub rows (attention path)")


@pytest.mark.parametrize("heads", [1, 8, 16])
def test_gat_tma_gather4_variant_is_bit_identical(heads):
    """K3 with the K|V rows of four neighbours fetched by one TMA tile::gather4 per round (K and V are column views of one
    buffer): same bits as the cp.async ring, which takes K and V in separate buffers.  Ragged rows, a hub row cut into
    slices, with and without the training statistics."""
    rs = np.random.RandomState(5)
    n, a = 3000, 128
    ei = random_graph(n, 40000, seed=6, isolated=5, hub=(17, 9000))
    from tf_geometric_b200 import _structure
    csr, _ = _structure.csr_for_edge_index(dev(ei, torch.int32), n, add_self_loop=True)
    q = dev(rs.randn(n, a).astype(np.float32))
    kv = dev(rs.randn(n, 2 * a).astype(np.float32))
    bias = dev(rs.randn(a).astype(np.float32))
    sep_k, sep_v = kv[:, :a].contiguous(), kv[:, a:].contiguous()
    want = ops.gat_fused(csr, q, sep_k, sep_v, heads, bias=bias, act=ops.ACT_RELU)
    got = ops.gat_fused(csr, q, kv[:, :a], kv[:, a:], heads, bias=bias, act=ops.ACT_RELU)
    assert torch.equal(got, want)
    want_out, want_stats = ops.gat_fused_stats(csr, q, sep_k, sep_v, heads, bias=bias, act=ops.ACT_RELU)
    got_out, got_stats = ops.gat_fused_stats(csr, q, kv[:, :a], kv[:, a:], heads, bias=bias, act=ops.ACT_RELU)
    assert torch.equal(got_out, want_out) and torch.equal(got_stats, want_stats)
