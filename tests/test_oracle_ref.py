"""CPU: the C restatement (oracle/geometry_ops.c) against the reference's OWN op kernels
(lmbspecialops/src/{warp2d,median3x3downsample,scaleinvariantgradient,leakyrelu,depthtoflow,depthtonormals}.cc, unmodified,
over oracle/ref_stub/).  Bit equality, edge cases included: this is what pins the oracle's warp2d /
scale_invariant_gradient / leaky_relu forward values, which no test of the reference holds.

The digests of the reference kernels' outputs on the inputs below (oracle.ref.output_digest: dtype, shape and bits) are
stored in tests/golden/reference_ops.json by tests/golden/make_reference_ops_golden.py, which runs them through
oracle/_ref/libref_ops.so; each case yields (golden key, op name, arguments), and the op name is the same function in
oracle.ops and oracle.ref."""
import json
import os

import numpy as np
import pytest

from oracle import ops as oops
from oracle import ref

TYPES = (np.float32, np.float64)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    both_nan = np.isnan(a) & np.isnan(b)          # a NaN is a NaN (payloads are not part of the contract)
    u = np.uint32 if a.dtype == np.float32 else np.uint64
    return bool(np.all(both_nan | (a.view(u) == b.view(u))))


def _k(*parts):
    return "/".join(p.__name__ if isinstance(p, type) else str(p) for p in parts)


def warp2d_cases(dtype, border_mode, normalized):
    rng = np.random.RandomState(11)
    inp = rng.uniform(-2, 2, (2, 3, 13, 17)).astype(dtype)
    scale = 0.3 if normalized else 4.0
    disp = rng.uniform(-scale, scale, (2, 2, 13, 17)).astype(dtype)
    # the cases that are easy to get wrong (SURVEY.md appendix A.5): p2 in (-1, 0) (truncation toward zero, negative
    # fractional weight), exact integers, the last row / column, NaN, +-inf, values beyond the int range
    disp[0, 0, 0, 0] = -0.5 / (17 if normalized else 1); disp[0, 1, 0, 0] = -0.25 / (13 if normalized else 1)
    disp[0, 0, 1, 1] = 0.0; disp[0, 1, 1, 1] = 0.0
    disp[0, 0, 12, 16] = 0.0; disp[0, 1, 12, 16] = 0.0
    disp[0, 0, 2, 3] = np.nan
    disp[0, 1, 3, 4] = np.nan
    disp[0, 0, 4, 5] = np.inf; disp[0, 1, 5, 6] = -np.inf
    disp[1, 0, 6, 7] = 3e9; disp[1, 1, 7, 8] = -3e9
    disp[1, 0, 8, 9] = 1e20; disp[1, 1, 9, 10] = -1e30
    yield _k("warp2d", dtype, border_mode, normalized), "warp2d", (inp, disp, normalized, border_mode, 0.375)


def warp2d_rank_cases(dtype):
    rng = np.random.RandomState(12)
    inp = rng.rand(5, 7).astype(dtype)                  # rank 2: C == 1, N == 1 (warp2d.cc:150-160)
    disp = rng.uniform(-2, 2, (2, 5, 7)).astype(dtype)
    yield _k("warp2d_rank2", dtype), "warp2d", (inp, disp)
    inp = rng.rand(2, 2, 3, 5, 7).astype(dtype)         # rank 5: leading dims collapse
    disp = rng.uniform(-2, 2, (2, 2, 2, 5, 7)).astype(dtype)
    yield _k("warp2d_rank5", dtype), "warp2d", (inp, disp, False, "value")


def median_cases(dtype):
    rng = np.random.RandomState(13)
    for shape in ((1, 1), (1, 5), (5, 1), (2, 3, 9, 12), (3, 10, 13), (4, 7)):
        yield _k("median", dtype, "x".join(map(str, shape))), "median3x3_downsample", (rng.rand(*shape).astype(dtype),)
    # ties, NaNs, infinities: the result depends on the exact compare / swap order of median3x3downsample.cc:133-177
    a = rng.randint(0, 3, (6, 12, 14)).astype(dtype)
    a[0, 3, 4] = np.nan; a[1, 0, 0] = np.nan; a[1, 0, 1] = np.nan; a[2, 5, 5] = np.inf; a[2, 6, 6] = -np.inf
    a[3, :, :] = np.where(rng.rand(12, 14) < 0.3, np.nan, a[3])
    yield _k("median", dtype, "ties"), "median3x3_downsample", (a,)


def scale_invariant_gradient_cases(dtype):
    rng = np.random.RandomState(14)
    a = rng.uniform(-3, 3, (2, 3, 11, 9)).astype(dtype)
    a[0, 0, 0, 0] = 0.0; a[0, 0, 0, 1] = -0.0; a[0, 1, 2, 2] = np.nan; a[1, 2, 3, 3] = np.inf
    for i, (deltas, weights, eps) in enumerate((((1,), (1.0,), 0.001), ((1, 2, 4, 8, 16), (1.0, 0.5, 0.25, 0.125, 0.0625), 0.01),
                                                ((-1, 3), (2.0, -1.5), 1e-3), ((20,), (1.0,), 1e-3))):
        yield _k("sig", dtype, i), "scale_invariant_gradient", (a, deltas, weights, eps)
    b = rng.rand(7, 5).astype(dtype)    # rank 2
    yield _k("sig", dtype, "rank2"), "scale_invariant_gradient", (b,)


def leaky_relu_cases(dtype):
    rng = np.random.RandomState(15)
    a = rng.uniform(-5, 5, (3, 4, 5)).astype(dtype)
    a.flat[:6] = [0.0, -0.0, np.nan, np.inf, -np.inf, np.finfo(dtype).tiny]
    for leak in (0.1, 0.0, 1.0, -0.5, 2.0):
        yield _k("leaky_relu", dtype, leak), "leaky_relu", (a, leak)


def depth_to_flow_cases(dtype, rotation_format, inverse_depth, normalize_flow):
    rng = np.random.RandomState(16)
    n = 3
    depth = rng.uniform(0.2, 4.0, (n, 1, 9, 12)).astype(dtype)
    depth[0, 0, 0, 0] = 0.0; depth[0, 0, 0, 1] = -1.0; depth[0, 0, 0, 2] = np.nan; depth[0, 0, 0, 3] = np.inf   # invalid branches
    intrinsics = np.tile(np.array([[0.89115971, 1.18821287, 0.5, 0.5]]), (n, 1)).astype(dtype)
    aa = rng.uniform(-0.3, 0.3, (n, 3)); aa[1] = 1e-8     # below the 1e-6 angle threshold: identity
    if rotation_format == "angleaxis3":
        rot = aa
    elif rotation_format == "quaternion":
        ang = np.linalg.norm(aa, axis=1, keepdims=True)
        rot = np.concatenate([np.cos(ang / 2), np.sin(ang / 2) * aa / np.maximum(ang, 1e-12)], axis=1) * 1.7   # un-normalised on purpose
    else:
        rot = oops.rotation_matrix(aa.astype(np.float64), "angleaxis3").reshape(n, 9)
    rot = rot.astype(dtype)
    t = rng.uniform(-1, 1, (n, 3)).astype(dtype)
    yield (_k("depth_to_flow", dtype, rotation_format, inverse_depth, normalize_flow), "depth_to_flow",
           (depth, intrinsics, rot, t, rotation_format, inverse_depth, normalize_flow))


def depth_to_normals_cases(dtype, inverse_depth):
    rng = np.random.RandomState(31)
    d = rng.uniform(0.2, 4.0, (2, 1, 17, 23)).astype(dtype)
    d[0, 0, 3, 4] = -1.0; d[0, 0, 8, 8] = 0.0; d[1, 0, 5, 5] = np.nan; d[1, 0, 9, 12] = np.inf; d[1, 0, 2, 20] = 1e-30
    K = np.array([[0.89115971, 1.18821287, 0.5, 0.5], [1.1, 0.9, 0.45, 0.55]], dtype)
    yield _k("depth_to_normals", dtype, inverse_depth), "depth_to_normals", (d, K, inverse_depth)


def reference_cases():
    """Every case whose reference output digest tests/golden/reference_ops.json holds."""
    for dt in TYPES:
        for flag in (False, True):
            yield from depth_to_normals_cases(dt, flag)
            for border_mode in ("clamp", "value"):
                yield from warp2d_cases(dt, border_mode, flag)
            for rotation_format in ("matrix", "quaternion", "angleaxis3"):
                for normalize_flow in (False, True):
                    yield from depth_to_flow_cases(dt, rotation_format, flag, normalize_flow)
        yield from warp2d_rank_cases(dt)
        yield from median_cases(dt)
        yield from scale_invariant_gradient_cases(dt)
        yield from leaky_relu_cases(dt)


@pytest.fixture(scope="module")
def reference(golden_dir):
    with open(os.path.join(golden_dir, "reference_ops.json")) as f:
        return json.load(f)


def check_cases(reference, cases):
    """Runs each case through the oracle and demands the reference kernel's bits; returns the oracle's outputs."""
    outs = []
    for key, op, args in cases:
        got = getattr(oops, op)(*args)
        assert ref.output_digest(got) == reference[key], key
        outs.append(got)
    return outs


@pytest.mark.skipif(not ref.available(), reason="needs oracle/_ref/libref_ops.so, built from the reference's op sources")
def test_ref_registers_the_reference_kernels():
    ks = ref.kernels()
    for op in ("Warp2d", "Median3x3Downsample", "ScaleInvariantGradient", "ScaleInvariantGradientGrad", "LeakyReluLmb",
               "LeakyReluLmbGrad", "DepthToFlow", "DepthToNormals"):
        for t in ("float", "double"):
            assert "%s/CPU/%s" % (op, t) in ks


@pytest.mark.parametrize("dtype", TYPES)
@pytest.mark.parametrize("border_mode", ("clamp", "value"))
@pytest.mark.parametrize("normalized", (False, True))
def test_warp2d_equals_reference_source(reference, dtype, border_mode, normalized):
    check_cases(reference, warp2d_cases(dtype, border_mode, normalized))


@pytest.mark.parametrize("dtype", TYPES)
def test_warp2d_rank_handling_equals_reference_source(reference, dtype):
    check_cases(reference, warp2d_rank_cases(dtype))


@pytest.mark.parametrize("dtype", TYPES)
def test_median_equals_reference_source(reference, dtype):
    check_cases(reference, median_cases(dtype))


@pytest.mark.parametrize("dtype", TYPES)
def test_scale_invariant_gradient_equals_reference_source(reference, dtype):
    check_cases(reference, scale_invariant_gradient_cases(dtype))


@pytest.mark.parametrize("dtype", TYPES)
def test_leaky_relu_equals_reference_source(reference, dtype):
    check_cases(reference, leaky_relu_cases(dtype))


@pytest.mark.parametrize("dtype", TYPES)
@pytest.mark.parametrize("rotation_format", ("matrix", "quaternion", "angleaxis3"))
@pytest.mark.parametrize("inverse_depth", (False, True))
@pytest.mark.parametrize("normalize_flow", (False, True))
def test_depth_to_flow_equals_reference_source(reference, dtype, rotation_format, inverse_depth, normalize_flow):
    (got,) = check_cases(reference, depth_to_flow_cases(dtype, rotation_format, inverse_depth, normalize_flow))
    assert got.shape == (3, 2, 9, 12)


@pytest.mark.parametrize("dtype", TYPES)
@pytest.mark.parametrize("inverse_depth", (False, True))
def test_depth_to_normals_equals_reference_source(reference, dtype, inverse_depth):
    """depthtonormals.cc compiled unmodified (Matrix3::inverse / cross / normalize from the stub) against the C restatement:
    borders, non-positive, zero, NaN and infinite depths, two cameras."""
    (a,) = check_cases(reference, depth_to_normals_cases(dtype, inverse_depth))
    assert a.shape == (2, 3, 17, 23)
    assert np.isnan(a[:, :, 0, :]).all() and np.isnan(a[:, :, :, -1]).all()          # border
    ok = ~np.isnan(a[:, 0])
    norms = np.sqrt((a ** 2).sum(axis=1))[ok]      # unit normals (a pixel whose two half-normals cancel stays at its tiny sum)
    assert ok.sum() > 100 and (np.abs(norms - 1.0) < 1e-5).mean() > 0.98


def test_depth_to_normals_of_a_fronto_parallel_plane_points_at_the_camera():
    d = np.full((1, 9, 11), 2.5, np.float32)
    n = oops.depth_to_normals(d, np.array([0.9, 1.2, 0.5, 0.5], np.float32))
    inner = n[0, :, 1:-1, 1:-1]
    assert np.allclose(inner[0], 0, atol=1e-6) and np.allclose(inner[1], 0, atol=1e-6) and np.allclose(np.abs(inner[2]), 1, atol=1e-6)
