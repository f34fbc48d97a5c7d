# coding=utf-8
"""K4 round 2 (tfgk_gemm_proj_f32): several projections of the same rows in one tcgen05 launch.
Checked against float64, and bit-for-bit against the single-projection tensor-core kernel (same 3xTF32 arithmetic, so the
fused launch must not change a single bit of Q, K, V or the GCN projection)."""
import numpy as np
import pytest
import torch

from tf_geometric_b200 import ops
from conftest import assert_close

pytestmark = pytest.mark.gpu


def dev(a):
    return ops.as_device(a)


def _blocks(rs, k, widths, m, with_bias=True):
    blocks, host = [], []
    for i, n in enumerate(widths):
        w = (rs.randn(k, n) / np.sqrt(k)).astype(np.float32)
        b = rs.randn(n).astype(np.float32) if with_bias and i % 2 == 0 else None
        act = ops.ACT_RELU if i % 3 == 0 else ops.ACT_NONE
        host.append((w, b, act))
        blocks.append((dev(w), None if b is None else dev(b), act, None))
    return blocks, host


@pytest.mark.parametrize("m,k,widths", [
    (4096, 100, [128, 128, 128]), (5000, 100, [128, 128, 128, 128]), (777, 100, [128]), (130000, 100, [128, 128, 128]),
    (3001, 128, [128, 64]), (1000, 33, [100, 7, 128]), (129, 8, [16]), (2708, 512, [16, 7]), (640, 20, [48, 128, 96, 1])])
def test_gemm_proj_matches_float64_and_single_projection_kernel(m, k, widths):
    rs = np.random.RandomState(m + k + len(widths))
    a = rs.randn(m, k).astype(np.float32)
    blocks, host = _blocks(rs, k, widths, m)
    outs = ops.gemm_proj(dev(a), blocks)
    for (w, b, act), got in zip(host, outs):
        want = a.astype(np.float64) @ w.astype(np.float64)
        if b is not None:
            want = want + b
        if act == ops.ACT_RELU:
            want = np.maximum(want, 0)
        assert_close(got.cpu().numpy(), want, rtol=1e-5, atol_scale=5e-6, what="gemm_proj block of width {}".format(w.shape[1]))
        single = ops.gemm(dev(a), dev(w), bias=None if b is None else dev(b), act=act)
        if k <= 512 and k % 4 == 0 and m * k >= (1 << 14):      # shapes the round-1 tensor-core kernel takes
            assert torch.equal(got, single), "fused launch changed bits (width {})".format(w.shape[1])


def test_gemm_proj_writes_column_slices_of_wider_buffers():
    rs = np.random.RandomState(3)
    m, k = 3000, 100
    a = rs.randn(m, k).astype(np.float32)
    wq, wk, wv = [(rs.randn(k, 128) / 10).astype(np.float32) for _ in range(3)]
    bq = rs.randn(128).astype(np.float32)
    q = torch.full((m, 128), 7.0, device="cuda")
    kv = torch.full((m, 256 + 4), 7.0, device="cuda")
    ops.gemm_proj(dev(a), [(dev(wq), dev(bq), ops.ACT_RELU, q), (dev(wk), None, ops.ACT_NONE, kv[:, :128]),
                           (dev(wv), None, ops.ACT_NONE, kv[:, 128:256])])
    a64 = a.astype(np.float64)
    assert_close(q.cpu().numpy(), np.maximum(a64 @ wq + bq, 0), rtol=1e-5, atol_scale=5e-6, what="Q")
    assert_close(kv[:, :128].cpu().numpy(), a64 @ wk, rtol=1e-5, atol_scale=5e-6, what="K")
    assert_close(kv[:, 128:256].cpu().numpy(), a64 @ wv, rtol=1e-5, atol_scale=5e-6, what="V")
    assert float((kv[:, 256:] - 7.0).abs().max()) == 0.0, "columns outside the blocks were touched"


def test_gemm_proj_row_blocks_at_different_addresses():
    """The partitioned path hands the kernel one base pointer per owner rank; here the parts are separate tensors on one
    GPU.  Any starting part gives the same bits as the contiguous matrix."""
    rs = np.random.RandomState(4)
    k, part_rows, n_parts, m = 100, 1280, 5, 5 * 1280 - 700      # last part is short
    a = rs.randn(n_parts * part_rows, k).astype(np.float32)
    parts = [dev(a[i * part_rows:(i + 1) * part_rows].copy()) for i in range(n_parts)]
    blocks, host = _blocks(rs, k, [128, 128, 40], m)
    want = ops.gemm_proj(dev(a[:m]), blocks)
    for first in (0, 3, 4):
        got = ops.gemm_proj(parts[0], [(w, b, act, None) for w, b, act, _ in blocks], a_parts=[p.data_ptr() for p in parts],
                            part_rows=part_rows, first_part=first, num_rows=m)
        for g, w_ in zip(got, want):
            assert g.shape[0] == m and torch.equal(g, w_)
    got = ops.gemm_proj(parts[0], [(w, b, act, None) for w, b, act, _ in blocks], a_parts=[p.data_ptr() for p in parts],
                        part_rows=part_rows, first_part=1, num_rows=m, max_ctas=24)
    for g, w_ in zip(got, want):
        assert torch.equal(g, w_)


def test_gat_layer_uses_one_projection_launch():
    import tf_geometric_b200 as tfg
    from tf_geometric_b200 import _ffi
    from conftest import random_graph
    rs = np.random.RandomState(0)
    n = 5000
    ei = dev(random_graph(n, 40000, seed=1, symmetric=True))
    x = dev(rs.randn(n, 100).astype(np.float32))
    layer = tfg.layers.GAT(128, num_heads=8, activation=tfg.nn.relu, seed=1)
    layer([x, ei])
    trace = _ffi.CallTrace()
    _ffi.set_trace(trace)
    try:
        layer([x, ei])
    finally:
        _ffi.set_trace(None)
    assert trace.counts.get("tfgk_gemm_proj_f32") == 1 and trace.counts.get("tfgk_gemm_f32", 0) == 0


def test_gemm_proj_transposed_weights_and_colsum():
    """dX = dY W^T on the tensor-core kernel (weights given as [n, K]) and the deterministic column sum used for db."""
    rs = np.random.RandomState(8)
    m, k = 7001, 128
    g = rs.randn(m, 2 * k).astype(np.float32)
    w1, w2 = (rs.randn(100, k) / 10).astype(np.float32), (rs.randn(60, k) / 10).astype(np.float32)
    gd = dev(g)
    d1, d2 = ops.gemm_proj(gd[:, :k], [(dev(w1), None, ops.ACT_NONE, None, True)])[0], \
        ops.gemm(gd[:, k:], dev(w2), trans_b=True)
    assert_close(d1.cpu().numpy(), g[:, :k].astype(np.float64) @ w1.T, rtol=1e-5, atol_scale=5e-6, what="dY W^T (gemm_proj)")
    assert_close(d2.cpu().numpy(), g[:, k:].astype(np.float64) @ w2.T, rtol=1e-5, atol_scale=5e-6, what="dY W^T (gemm)")
    for view in (gd, gd[:, :k], gd[:, 3:40]):
        got = ops.colsum(view)
        assert_close(got.cpu().numpy(), view.cpu().numpy().astype(np.float64).sum(0), rtol=1e-5, atol_scale=2e-6, what="colsum")
        assert torch.equal(got, ops.colsum(view))


@pytest.mark.parametrize("m,k,widths", [(4096, 100, [128, 128, 128]), (130000, 100, [128, 128, 128, 128]), (777, 100, [128]),
                                        (3001, 128, [128, 64]), (1000, 33, [100, 7, 128]), (129, 8, [16]), (5000, 300, [128])])
def test_gemm_proj_tensor_memory_operand_variant(m, k, widths):
    """The projection kernel: the split A operands are staged in tensor memory (tcgen05.st) and the MMAs read A from there.
    fp32-accurate against float64 for every shape, and repeatable bit for bit."""
    rs = np.random.RandomState(m + k)
    a = rs.randn(m, k).astype(np.float32)
    blocks, host = _blocks(rs, k, widths, m)
    got = ops.gemm_proj(dev(a), blocks)
    again = ops.gemm_proj(dev(a), blocks)
    for (w, b, act), g, g2 in zip(host, got, again):
        ref = a.astype(np.float64) @ w.astype(np.float64)
        if b is not None:
            ref = ref + b
        if act == ops.ACT_RELU:
            ref = np.maximum(ref, 0)
        assert_close(g.cpu().numpy(), ref, rtol=1e-5, atol_scale=5e-6, what="ts gemm_proj width {}".format(w.shape[1]))
        assert torch.equal(g, g2), "gemm_proj is not repeatable (width {})".format(w.shape[1])
