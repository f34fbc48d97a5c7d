# coding=utf-8
"""K4 tensor-core path (tcgen05, 3xTF32 split): fp32-level accuracy against float64, far inside the 1e-4 gate that a
single TF32 pass would miss.  Shapes cover the projections of the hot path and the ragged edges (M, N, K tails)."""
import numpy as np
import pytest
import torch

from tf_geometric_b200 import ops
from conftest import assert_close

pytestmark = pytest.mark.gpu


def dev(a):
    return ops.as_device(a)


@pytest.mark.parametrize("m,n,k", [
    (128, 128, 32), (128, 16, 8), (4096, 128, 100), (5000, 128, 128), (2708, 16, 512), (3000, 7, 16),
    (1000, 64, 20), (777, 200, 333), (130000, 128, 100), (300, 256, 64), (129, 48, 5)])
def test_gemm_tc_matches_float64(m, n, k):
    rs = np.random.RandomState(m + n + k)
    a = rs.randn(m, k).astype(np.float32)
    b = (rs.randn(k, n) / np.sqrt(k)).astype(np.float32)
    bias = rs.randn(n).astype(np.float32)
    want = a.astype(np.float64) @ b.astype(np.float64)
    got = ops.gemm(dev(a), dev(b)).cpu().numpy()
    err = np.abs(got - want).max() / np.abs(want).max()
    assert err < 5e-6, "3xTF32 relative error {:.2e} (single-pass TF32 would be ~1e-3)".format(err)
    got = ops.gemm(dev(a), dev(b), bias=dev(bias), act=ops.ACT_RELU).cpu().numpy()
    assert_close(got, np.maximum(want + bias, 0), rtol=1e-5, atol_scale=5e-6, what="tc gemm + bias + relu")


def test_gemm_tc_strided_operands_and_output_slices():
    rs = np.random.RandomState(0)
    m, k, n = 3000, 100, 128
    big_a = rs.randn(m, 3 * k + 4).astype(np.float32)          # lda = 304
    a = dev(big_a)[:, 4:4 + k]                                  # 16-byte aligned column offset
    b = dev((rs.randn(k, n) / 10).astype(np.float32))
    out = torch.zeros((m, 2 * n), dtype=torch.float32, device="cuda")
    ops.gemm(a, b, out=out[:, n:])
    want = big_a[:, 4:4 + k].astype(np.float64) @ b.cpu().numpy().astype(np.float64)
    assert_close(out[:, n:].cpu().numpy(), want, rtol=1e-5, atol_scale=5e-6, what="strided tc gemm")
    assert float(out[:, :n].abs().max()) == 0.0
    a2 = dev(big_a)[:, 1:1 + k]                                  # unaligned column offset -> scalar-load variant
    ops.gemm(a2, b, out=out[:, :n])
    want2 = big_a[:, 1:1 + k].astype(np.float64) @ b.cpu().numpy().astype(np.float64)
    assert_close(out[:, :n].cpu().numpy(), want2, rtol=1e-5, atol_scale=5e-6, what="unaligned tc gemm")


def test_gemm_tc_is_deterministic():
    rs = np.random.RandomState(1)
    a, b = dev(rs.randn(20000, 100).astype(np.float32)), dev(rs.randn(100, 128).astype(np.float32))
    first = ops.gemm(a, b)
    for _ in range(3):
        assert torch.equal(first, ops.gemm(a, b))
