# coding=utf-8
"""GPU parity for the pooling family beyond the plain segment reductions (SURVEY.md 8(f)2): radix argsort building
blocks, topk_pool, set2set (attention read-out on the fused kernel), induced subgraphs / BatchGraph and sag_pool.
Integer outputs are compared bit for bit with the oracle; the reference's own outputs are in
tests/golden/ref_exec_pool2.npz (replayed by test_gpu_golden.py)."""
import numpy as np
import pytest
import torch

import tf_geometric_b200 as tfg
from tf_geometric_b200 import ops
from oracle import tfg_oracle as o
from conftest import random_graph, assert_close, glorot
import golden_cases

pytestmark = pytest.mark.gpu


def dev(a, dtype=None):
    return ops.as_device(a, dtype)


def host(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def test_sort_keys_and_stable_argsort():
    rs = np.random.RandomState(0)
    x = np.concatenate([rs.randn(20000), [0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 3.5, 3.5, 3.5],
                        np.round(rs.randn(5000), 1)]).astype(np.float32)
    x = x[rs.permutation(len(x))]
    for descending in (False, True):
        perm = host(ops.stable_argsort(ops.sort_keys_f32(dev(x), descending=descending)))
        want = np.argsort(-(x + np.float32(0)) if descending else x + np.float32(0), kind="stable")
        np.testing.assert_array_equal(perm, want)
    keys = rs.randint(0, 1 << 16, 70000).astype(np.int32)
    np.testing.assert_array_equal(host(ops.stable_argsort(dev(keys), key_bits=16)), np.argsort(keys, kind="stable"))
    wide = rs.randint(-2 ** 31, 2 ** 31 - 1, 30000, dtype=np.int64).astype(np.int32)
    np.testing.assert_array_equal(host(ops.stable_argsort(dev(wide))), np.argsort(wide.view(np.uint32), kind="stable"))
    assert host(ops.stable_argsort(dev(np.zeros(0, np.int32)))).shape == (0,)


@pytest.mark.parametrize("k,ratio", [(1, None), (7, None), (100000, None), (None, 0.25), (None, 0.5), (None, 1.0)])
def test_topk_pool_matches_oracle(k, ratio):
    rs = np.random.RandomState(5)
    n, sources = 60000, 400
    src = rs.randint(0, sources, n).astype(np.int32)
    src[src == 17] = 18                                               # an empty source
    src[:5] = sources - 1
    score = np.round(rs.randn(n), 2).astype(np.float32)               # plenty of ties
    got = host(tfg.nn.topk_pool(dev(src), dev(score), k=k, ratio=ratio))
    want = o.topk_pool(src, score, k=k, ratio=ratio)
    np.testing.assert_array_equal(got, want)
    assert got.dtype == np.int32
    sel_src = src[got]
    assert (np.diff(sel_src) >= 0).all()                              # grouped by ascending source
    same = np.diff(sel_src) == 0
    assert (np.diff(score[got])[same] <= 0).all()                     # best score first inside a source
    with pytest.raises(Exception):
        tfg.nn.topk_pool(dev(src), dev(score))
    with pytest.raises(Exception):
        tfg.nn.topk_pool(dev(src), dev(score), k=1, ratio=0.5)


@pytest.mark.parametrize("d,graphs,n", [(6, 9, 200), (64, 40, 5000), (64, 8, 4000), (128, 3, 9000)])
def test_set2set_matches_oracle(d, graphs, n):
    rs = np.random.RandomState(d)
    gi = np.sort(rs.randint(0, graphs, n)).astype(np.int32)
    gi[-1] = graphs - 1
    if d == 128:
        gi[: n * 2 // 3] = 0                                          # one graph with > 2048 nodes: a hub row
        gi = np.sort(gi)
    x = (rs.randn(n, d) * 0.5).astype(np.float32)
    k, r, b = glorot(rs, 2 * d, 4 * d), glorot(rs, d, 4 * d), (rs.randn(4 * d) * 0.1).astype(np.float32)
    want = o.set2set(x, gi, o.numpy_lstm(k, r, b), 3)
    api = golden_cases.ProductApi()
    got = tfg.nn.set2set(dev(x), dev(gi), api.lstm(k, r, b), 3)
    assert_close(host(got), want, what="set2set d={}".format(d))
    layer = tfg.layers.Set2Set(num_iterations=2)
    out = layer([dev(x), dev(gi)])
    assert tuple(out.shape) == (graphs, 2 * d)
    np.testing.assert_array_equal(host(layer([dev(x), dev(gi)])), host(out))


def test_induced_subgraph_and_batch_graph():
    rs = np.random.RandomState(9)
    n = 3000
    ei = random_graph(n, 40000, seed=10)
    w = rs.rand(ei.shape[1]).astype(np.float32)
    x = rs.randn(n, 5).astype(np.float32)
    y = rs.randint(0, 7, n)
    gi = np.sort(rs.randint(0, 12, n)).astype(np.int32)
    keep = rs.permutation(n)[:1100].astype(np.int32)
    wx, wei, ww, wgi, wy = o.sample_new_graph_by_node_index(x, ei, w, keep, gi, y)
    batch = tfg.BatchGraph(x, ei, gi, None, y=y, edge_weight=w)
    for g, on_device in ((batch.to_device(), True), (batch, False)):
        sub = g.sample_new_graph_by_node_index(dev(keep) if on_device else keep)
        assert isinstance(sub, tfg.BatchGraph) and torch.is_tensor(sub.edge_index) == on_device
        np.testing.assert_array_equal(host(sub.x), wx)
        np.testing.assert_array_equal(host(sub.edge_index), wei)
        np.testing.assert_array_equal(host(sub.edge_weight), ww)
        np.testing.assert_array_equal(host(sub.node_graph_index), wgi)
        np.testing.assert_array_equal(host(sub.y), wy)
    plain = tfg.Graph(x, ei, edge_weight=w).to_device().sample_new_graph_by_node_index(dev(keep))
    assert type(plain) is tfg.Graph
    np.testing.assert_array_equal(host(plain.edge_index), wei)

    # from_graphs / to_graphs round trip on the device, with an interleaved (unsorted) batch in between
    parts = []
    for i, size in enumerate((5, 1, 9, 4)):
        pe = random_graph(size, 3 * size, seed=20 + i) if size > 1 else np.zeros((2, 0), np.int32)
        parts.append(tfg.Graph(rs.randn(size, 3).astype(np.float32), pe, y=np.arange(size) + 100 * i,
                               edge_weight=rs.rand(pe.shape[1]).astype(np.float32)).to_device())
    bg = tfg.BatchGraph.from_graphs(parts)
    assert bg.num_graphs == 4 and bg.num_nodes == 19
    np.testing.assert_array_equal(host(bg.node_graph_index), np.repeat(np.arange(4), [5, 1, 9, 4]))
    shuffle_n, shuffle_e = rs.permutation(bg.num_nodes), rs.permutation(bg.num_edges)
    inv = np.empty_like(shuffle_n)
    inv[shuffle_n] = np.arange(len(shuffle_n))
    mixed = tfg.BatchGraph(host(bg.x)[shuffle_n], inv[host(bg.edge_index)[:, shuffle_e]],
                           host(bg.node_graph_index)[shuffle_n], host(bg.edge_graph_index)[shuffle_e],
                           y=host(bg.y)[shuffle_n], edge_weight=host(bg.edge_weight)[shuffle_e]).to_device()
    ordered = mixed.reorder()
    assert (np.diff(host(ordered.node_graph_index)) >= 0).all() and (np.diff(host(ordered.edge_graph_index)) >= 0).all()
    back = bg.to_graphs()
    for a, b_ in zip(parts, back):
        np.testing.assert_array_equal(host(a.x), host(b_.x))
        np.testing.assert_array_equal(host(a.edge_index), host(b_.edge_index))
        np.testing.assert_array_equal(host(a.edge_weight), host(b_.edge_weight))
        np.testing.assert_array_equal(host(a.y), host(b_.y))


@pytest.mark.parametrize("k,ratio", [(3, None), (None, 0.4)])
def test_sag_pool_matches_oracle(k, ratio):
    rs = np.random.RandomState(31)
    n, graphs = 1500, 25
    ei = random_graph(n, 12000, seed=32, symmetric=True)
    w = (rs.rand(ei.shape[1]) + 0.1).astype(np.float32)
    x = rs.randn(n, 8).astype(np.float32)
    gi = np.sort(rs.randint(0, graphs, n)).astype(np.int32)
    gi[-1] = graphs - 1
    score_gnn = tfg.layers.GCN(1, seed=3)
    xd, eid, wd, gid = dev(x), dev(ei, torch.int32), dev(w), dev(gi)
    px, pei, pw, pgi = tfg.nn.sag_pool(xd, eid, wd, gid, score_gnn, k=k, ratio=ratio, score_activation=torch.tanh)
    scores = host(score_gnn([xd, eid, wd]))                             # feed the SAME scores to the oracle
    wx, wei, ww, wgi = o.sag_pool(x, ei, w, gi, lambda inputs: scores, k=k, ratio=ratio, score_activation=np.tanh)
    np.testing.assert_array_equal(host(pei), wei)
    np.testing.assert_array_equal(host(pgi), wgi)
    np.testing.assert_array_equal(host(pw), ww)
    assert_close(host(px), wx, rtol=1e-6, atol_scale=1e-6, what="pooled x")
    layer = tfg.layers.SAGPool(score_gnn, k=k, ratio=ratio, score_activation=torch.tanh)
    lx, lei, lw, lgi = layer([xd, eid, wd, gid])
    np.testing.assert_array_equal(host(lei), wei)
    np.testing.assert_array_equal(host(lx), host(px))
    pooled = tfg.layers.MaxPool()([lx, lgi])
    assert tuple(pooled.shape) == (graphs, 8)
    np.testing.assert_array_equal(host(pooled), host(tfg.nn.max_pool(lx, lgi)))
    np.testing.assert_array_equal(host(tfg.layers.MeanPool()([lx, lgi, graphs])), host(tfg.nn.mean_pool(lx, lgi, graphs)))


def test_pools_over_few_large_graphs_use_edge_sized_tasks():
    """Average segment length >= 128: the work plan shrinks its tasks from 32 rows to ~512 entries (ops.build_plan);
    per-graph sums stay sequential, so the results are still bit-exact."""
    rs = np.random.RandomState(77)
    n, graphs, d = 12000, 20, 24
    gi = np.sort(rs.randint(0, graphs, n)).astype(np.int32)
    gi[-1] = graphs - 1
    x = rs.randn(n, d).astype(np.float32)
    from tf_geometric_b200 import _structure
    seg = _structure.csr_for_segment_ids(dev(gi), graphs)
    if seg.rowptr.is_cuda:         # built by the kernels; the CPU test double (also used on GPU hosts) builds no plan
        assert seg.plan is not None and seg.plan.n_hubs == 0 and seg.plan.n_tasks >= graphs
    for name in ("mean_pool", "sum_pool", "max_pool", "min_pool"):
        got = host(getattr(tfg.nn, name)(dev(x), dev(gi), graphs))
        np.testing.assert_array_equal(got, getattr(o, name)(x, gi, graphs), err_msg=name)


def test_sort_pool_drop_edge_layer_and_map_reduce_layer():
    rs = np.random.RandomState(55)
    n, graphs = 2000, 30
    ei = random_graph(n, 15000, seed=56, symmetric=True)
    w = rs.rand(ei.shape[1]).astype(np.float32)
    x = rs.randn(n, 6).astype(np.float32)
    gi = np.sort(rs.randint(0, graphs, n)).astype(np.int32)
    gi[-1] = graphs - 1
    xd, eid, wd, gid = dev(x), dev(ei, torch.int32), dev(w), dev(gi)
    # SortPool: rank by the last feature column
    keep = o.topk_pool(gi, x[:, -1], k=10)
    wx, wei, ww, wgi, _ = o.sample_new_graph_by_node_index(x, ei, w, keep, gi)
    px, pei, pw, pgi = tfg.layers.SortPool(k=10)([xd, eid, wd, gid])
    np.testing.assert_array_equal(host(px), wx)
    np.testing.assert_array_equal(host(pei), wei)
    np.testing.assert_array_equal(host(pw), ww)
    np.testing.assert_array_equal(host(pgi), wgi)
    keep = o.topk_pool(gi, x[:, 2], ratio=0.3)
    px, pei, _, _ = tfg.nn.sort_pool(xd, eid, wd, gid, ratio=0.3, sort_index=2)
    np.testing.assert_array_equal(host(px), x[keep])
    np.testing.assert_array_equal(host(pei), o.sample_new_graph_by_node_index(x, ei, w, keep)[1])

    # DropEdge layer
    layer = tfg.layers.DropEdge(rate=0.4, force_undirected=True)
    out = layer([eid, wd], training=True, seed=8)
    want = o.drop_edge([ei, w], 0.4, True, True, seed=8)
    np.testing.assert_array_equal(host(out[0]), want[0])
    np.testing.assert_array_equal(host(out[1]), want[1])
    same = layer([eid, wd], training=False)
    assert same[0] is eid and same[1] is wd
    with pytest.raises(ValueError):
        tfg.layers.DropEdge(rate=1.2)

    # MapReduceGNN: a user-defined mapper with a stock reducer
    class Doubler(tfg.layers.MapReduceGNN):
        def map(self, repeated_x, neighbor_x, edge_weight=None):
            return neighbor_x * 2.0 * edge_weight.unsqueeze(1)

        def reduce(self, neighbor_msg, node_index, num_nodes=None):
            return tfg.nn.mean_reducer(neighbor_msg, node_index, num_nodes)

        def update(self, x, reduced_neighbor_msg):
            return x + reduced_neighbor_msg

    got = Doubler()([xd, eid, wd])
    want = o.aggregate_neighbors(x, ei, w, lambda rx, nx, edge_weight=None: (nx * np.float32(2.0) * edge_weight[:, None]).astype(np.float32),
                                 o.mean_reducer, o.sum_updater, num_nodes=n)
    assert_close(host(got), want, rtol=1e-6, atol_scale=1e-6, what="MapReduceGNN")


def _torch_lstm(k, r, b):
    """The LSTM cell of oracle.numpy_lstm on torch tensors of any dtype/device (differentiable)."""
    units = r.shape[0]

    def lstm(inputs, initial_state=None, training=None):
        h, c = initial_state
        seq = []
        for t in range(inputs.shape[1]):
            z = inputs[:, t] @ k + h @ r + b
            i, f, g, o_ = (z[:, j * units:(j + 1) * units] for j in range(4))
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
            h = torch.sigmoid(o_) * torch.tanh(c)
            seq.append(h)
        return torch.stack(seq, dim=1), h, c
    return lstm


@pytest.mark.parametrize("d,graphs,n", [(6, 7, 150), (64, 5, 3000)])
def test_set2set_gradients_match_autodiff(d, graphs, n):
    from oracle import torch_cpu_port as port
    rs = np.random.RandomState(d + 1)
    gi = np.sort(rs.randint(0, graphs, n)).astype(np.int32)
    gi[-1] = graphs - 1
    x = (rs.randn(n, d) * 0.5).astype(np.float32)
    k, r, b = glorot(rs, 2 * d, 4 * d), glorot(rs, d, 4 * d), (rs.randn(4 * d) * 0.1).astype(np.float32)
    gout = rs.randn(graphs, 2 * d).astype(np.float32)

    tp = [dev(a).requires_grad_(True) for a in (x, k, r, b)]
    y = tfg.nn.set2set(tp[0], dev(gi), _torch_lstm(*tp[1:]), 2)
    (y * dev(gout)).sum().backward()

    t64 = [torch.tensor(a.astype(np.float64), requires_grad=True) for a in (x, k, r, b)]
    ids = torch.from_numpy(gi.astype(np.int64))
    lstm64 = _torch_lstm(*t64[1:])
    h = torch.zeros((graphs, 2 * d), dtype=torch.float64)
    state = [torch.zeros((1, d), dtype=torch.float64), torch.zeros((1, d), dtype=torch.float64)]
    for _ in range(2):                                                   # set2set.py:28-40 on float64 torch ops
        q, sh, sc = lstm64(h.unsqueeze(0), initial_state=state)
        state = [sh, sc]
        q = q.squeeze(0)
        score = (t64[0] * q.index_select(0, ids)).sum(-1)
        a = port.segment_softmax(score, ids, graphs)
        att_h = torch.zeros((graphs, d), dtype=torch.float64).index_add_(0, ids, t64[0] * a.unsqueeze(1))
        h = torch.cat([q, att_h], dim=-1)
    (h * torch.tensor(gout.astype(np.float64))).sum().backward()

    assert_close(host(y), h.detach().numpy(), what="set2set forward (training path)")
    for name, mine, ref in zip(("x", "lstm kernel", "lstm recurrent kernel", "lstm bias"), tp, t64):
        assert mine.grad is not None, name
        assert_close(host(mine.grad), ref.grad.numpy(), rtol=1e-3, atol_scale=2e-4, what="set2set d " + name)
    layer = tfg.layers.Set2Set(num_iterations=2, trainable=True)
    out = layer([dev(x), dev(gi)])
    out.sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in layer.parameters())
