"""GPU: the training-side companions (SURVEY.md section 8 f4) against the reference's own CPU kernels
(scaleinvariantgradient.cc, leakyrelu.cc, replacenonfinite.cc, depthtonormals.cc, unmodified): bit exact, same IEEE
operations in the same order.  The digests of the reference kernels' outputs on the inputs below
(oracle.ref.output_digest: dtype, shape and bits) are stored in tests/golden/reference_ops.json
(tests/golden/make_reference_ops_golden.py); each case yields (golden key, op name, arguments), and the op name is the
same function in demon_b200.lmbspecialops and oracle.ref."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.ref import output_digest

pytestmark = pytest.mark.gpu

TYPES = (np.float32, np.float64)


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    from demon_b200 import lmbspecialops
    return lmbspecialops


@pytest.fixture(scope="module")
def reference(golden_dir):
    with open(os.path.join(golden_dir, "reference_ops.json")) as f:
        return json.load(f)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    u = np.uint32 if a.dtype == np.float32 else np.uint64
    return bool(np.all((np.isnan(a) & np.isnan(b)) | (a.view(u) == b.view(u))))


def sig_grad_cases(dtype):
    rng = np.random.RandomState(21)
    x = rng.uniform(-3, 3, (3, 2, 19, 23)).astype(dtype)
    x[0, 0, 0, 0] = 0.0; x[0, 1, 3, 3] = np.nan; x[1, 0, 5, 5] = np.inf; x[2, 1, 7, 7] = -0.0
    for i, (deltas, weights, eps) in enumerate((((1,), (1.0,), 0.001), ((1, 2, 4, 8, 16), (1.0, 0.5, 0.25, 0.125, 0.0625), 0.01),
                                                ((-2, 3), (2.0, -1.5), 1e-3))):
        g = rng.uniform(-1, 1, (6, 2, 19, 23)).astype(dtype)
        yield "sig_grad/%s/%d" % (dtype.__name__, i), "scale_invariant_gradient_grad", (g, x, deltas, weights, eps)


def leaky_relu_grad_and_replace_nonfinite_cases(dtype):
    rng = np.random.RandomState(22)
    x = rng.uniform(-4, 4, (5, 7, 9)).astype(dtype)
    x.flat[:6] = [0.0, -0.0, np.nan, np.inf, -np.inf, 1e-30]
    g = rng.uniform(-1, 1, x.shape).astype(dtype)
    for leak in (0.1, 0.0, 1.5, -0.5):
        yield "leaky_relu_grad/%s/%r" % (dtype.__name__, leak), "leaky_relu_grad", (g, x, leak)
    for value in (0.0, -7.5):
        yield "replace_nonfinite/%s/%r" % (dtype.__name__, value), "replace_nonfinite", (x, value)
    yield "replace_nonfinite_grad/%s" % dtype.__name__, "replace_nonfinite_grad", (g, x)


def depth_to_normals_cases(dtype, inverse_depth):
    rng = np.random.RandomState(33)
    d = rng.uniform(0.2, 4.0, (3, 1, 37, 141)).astype(dtype)
    d[0, 0, 3, 4] = -1.0; d[0, 0, 8, 8] = 0.0; d[1, 0, 5, 5] = np.nan; d[2, 0, 9, 12] = np.inf
    K = np.array([[0.89115971, 1.18821287, 0.5, 0.5], [1.1, 0.9, 0.45, 0.55], [0.7, 0.7, 0.5, 0.4]], dtype)
    yield "gpu_depth_to_normals/%s/%s" % (dtype.__name__, inverse_depth), "depth_to_normals", (d, K, inverse_depth)


def reference_cases():
    """Every case whose reference output digest tests/golden/reference_ops.json holds."""
    for dt in TYPES:
        yield from sig_grad_cases(dt)
        yield from leaky_relu_grad_and_replace_nonfinite_cases(dt)
        for inverse_depth in (False, True):
            yield from depth_to_normals_cases(dt, inverse_depth)


@pytest.mark.parametrize("dtype", TYPES)
def test_sig_grad_equals_reference_source(ops, reference, dtype):
    for key, op, (g, x, deltas, weights, eps) in sig_grad_cases(dtype):
        got = getattr(ops, op)(g, x, deltas, weights, eps)
        assert got.shape == x.shape
        assert output_digest(got) == reference[key], key


@pytest.mark.parametrize("dtype", TYPES)
def test_leaky_relu_grad_and_replace_nonfinite_equal_reference_source(ops, reference, dtype):
    for key, op, args in leaky_relu_grad_and_replace_nonfinite_cases(dtype):
        assert output_digest(getattr(ops, op)(*args)) == reference[key], key


def test_sig_autograd_matches_numeric_gradient(ops):
    """The reference's own test of this op is analytic-vs-numeric (test_ScaleInvariantGradient.py:31-63); same here through
    torch.autograd in float64."""
    rng = np.random.RandomState(23)
    x = torch.from_numpy(rng.uniform(0.5, 2.0, (1, 1, 6, 7))).cuda().requires_grad_(True)
    deltas, weights, eps = (1, 2), (1.0, 0.5), 0.001
    w = torch.from_numpy(rng.uniform(-1, 1, (1, 2, 6, 7))).cuda()
    loss = (ops.scale_invariant_gradient_autograd(x, deltas, weights, eps) * w).sum()
    loss.backward()
    analytic = x.grad.cpu().numpy()
    xn = x.detach().cpu().numpy()
    num = np.zeros_like(xn)
    h = 1e-6
    for idx in np.ndindex(*xn.shape):
        xp, xm = xn.copy(), xn.copy()
        xp[idx] += h; xm[idx] -= h
        fp = (ops.scale_invariant_gradient(xp, deltas, weights, eps) * w.cpu().numpy()).sum()
        fm = (ops.scale_invariant_gradient(xm, deltas, weights, eps) * w.cpu().numpy()).sum()
        num[idx] = (fp - fm) / (2 * h)
    np.testing.assert_allclose(analytic, num, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("dtype", TYPES)
@pytest.mark.parametrize("inverse_depth", (False, True))
def test_depth_to_normals_equals_reference_source(ops, reference, dtype, inverse_depth):
    """depth_to_normals (v2 losses / blocks): bit exact against depthtonormals.cc, invalid depths and borders included;
    [4] intrinsics broadcast; rank rules of the op's shape function."""
    ((key, op, (d, K, _)),) = depth_to_normals_cases(dtype, inverse_depth)
    got = getattr(ops, op)(d, K, inverse_depth)
    assert got.shape == (3, 3, 37, 141) and output_digest(got) == reference[key], key
    one = ops.depth_to_normals(d[0, 0], K[0], inverse_depth)                      # rank 2 depth, [4] intrinsics
    assert one.shape == (1, 3, 37, 141) and bits_equal(one, got[:1])
    with pytest.raises(ValueError):
        ops.depth_to_normals(np.ones(5, dtype), K[0])
    with pytest.raises(ValueError):
        ops.depth_to_normals(d, np.ones((3, 3), dtype))
