"""ORACLE (test infrastructure) -- the reference's OWN CPU op kernels, compiled from the reference checkout's
lmbspecialops/src/{warp2d,median3x3downsample,scaleinvariantgradient,leakyrelu,depthtoflow,replacenonfinite,depthtonormals}.cc
(REF_SRC; unmodified, read where they lie) against the stub TensorFlow / Eigen headers in oracle/ref_stub/, as
oracle/_ref/libref_ops.so (git-ignored).

This is what pins the C restatement (oracle/geometry_ops.c) and the CUDA ops: tests/golden/make_reference_ops_golden.py
stores the digests of these kernels' outputs on the edge cases of tests/test_oracle_ref.py and
tests/test_gpu_training_ops.py (NaN / huge displacements, borders, ties, invalid depths), and those tests demand bit
equality with them.  The signatures mirror the reference's Python binding like oracle/ops.py does.  `available()` is
False where neither the library nor the reference sources exist.  Only tests/, __graft_entry__ and bench.py's CPU legs
may import this module.
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_ref", "libref_ops.so")
REF_SRC = "/root/reference/lmbspecialops/src"
_SOURCES = ["warp2d.cc", "median3x3downsample.cc", "scaleinvariantgradient.cc", "leakyrelu.cc", "depthtoflow.cc", "replacenonfinite.cc", "depthtonormals.cc"]


def build(force=False):
    """Compile _ref/libref_ops.so if the reference tree is present; returns the path or None."""
    have_src = all(os.path.isfile(os.path.join(REF_SRC, s)) for s in _SOURCES)
    if not have_src:
        return _LIB_PATH if os.path.isfile(_LIB_PATH) else None
    deps = [os.path.join(REF_SRC, s) for s in _SOURCES] + [os.path.join(_HERE, f) for f in (
        "ref_harness.cc", "ref_stub/tf_stub.h", "ref_stub/eigen_stub.h", "Makefile")]
    if force or not os.path.isfile(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "ref"])   # this function decided it is stale (make does not see Makefile edits)
    return _LIB_PATH


_lib = None


def available():
    return build() is not None


def lib():
    global _lib
    if _lib is None:
        path = build()
        if path is None:
            raise RuntimeError("oracle/_ref/libref_ops.so is not built and /root/reference is absent")
        _lib = ctypes.CDLL(path)
        _lib.ref_run.restype = ctypes.c_int
    return _lib


def kernels():
    buf = ctypes.create_string_buffer(4096)
    lib().ref_list(buf, 4096)
    return sorted(k for k in buf.value.decode().split(";") if k)


def run(op, inputs, attrs="", out_elems=None):
    """Run the reference CPU kernel `op` on numpy inputs (all float32 or all float64)."""
    arrs = [np.ascontiguousarray(a) for a in inputs]
    dt = arrs[0].dtype
    if dt not in (np.float32, np.float64) or any(a.dtype != dt for a in arrs):
        raise TypeError("reference kernels take float32 or float64 tensors of one type")
    n = len(arrs)
    data = (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrs])
    shapes = [d for a in arrs for d in a.shape]
    shapes_c = (ctypes.c_int64 * max(1, len(shapes)))(*shapes)
    ranks = (ctypes.c_int * n)(*[a.ndim for a in arrs])
    cap = int(out_elems if out_elems is not None else 4 * max(a.size for a in arrs) + 16)
    out = np.empty(cap, dtype=dt)
    oshape = (ctypes.c_int64 * 8)()
    orank = ctypes.c_int(0)
    err = ctypes.create_string_buffer(512)
    rc = lib().ref_run(op.encode(), int(dt == np.float64), attrs.encode(), n, data, shapes_c, ranks,
                       out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(cap), oshape, ctypes.byref(orank), err, 512)
    if rc != 0:
        raise RuntimeError("reference kernel %s: %s" % (op, err.value.decode()))
    shape = tuple(oshape[i] for i in range(orank.value))
    return out[:int(np.prod(shape)) if shape else 1].reshape(shape).copy()


def output_digest(a):
    """'<dtype>[<shape>]:<sha256 of the bits>' of an op output, every NaN replaced by the canonical quiet NaN first (NaN
    payloads are not part of the ops' contract).  Equal digests mean bit-equal outputs; tests/golden/reference_ops.json
    holds the digests of the reference kernels' outputs."""
    a = np.array(a, order="C", copy=True)
    a[np.isnan(a)] = np.nan
    return "%s%s:%s" % (a.dtype.name, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest())


def _b(v):
    return "1" if v else "0"


def warp2d(input, displacements, normalized=False, border_mode="clamp", border_value=0.0):
    """Warp2dOp::Compute, warp2d.cc:141-256."""
    return run("Warp2d", [input, displacements],
               "normalized:b=%s;border_mode:s=%s;border_value:f=%r" % (_b(normalized), border_mode, float(border_value)))


def median3x3_downsample(input):
    """Median3x3DownsampleOp::Compute, median3x3downsample.cc:83-184."""
    return run("Median3x3Downsample", [input])


def leaky_relu(input, leak=0.1):
    """LeakyReluLmbOp::Compute, leakyrelu.cc:62-82."""
    return run("LeakyReluLmb", [input], "leak:f=%r" % float(leak))


def leaky_relu_grad(gradients, input, leak=0.1):
    """LeakyReluLmbGradOp::Compute, leakyrelu.cc:127-155."""
    return run("LeakyReluLmbGrad", [gradients, input], "leak:f=%r" % float(leak))


def _sig_attrs(deltas, weights, epsilon):
    return "deltas:li=%s;weights:lf=%s;epsilon:f=%r" % (",".join(str(int(d)) for d in deltas),
                                                     ",".join(repr(float(w)) for w in weights), float(epsilon))


def scale_invariant_gradient(input, deltas=(1,), weights=(1.0,), epsilon=0.001):
    """ScaleInvariantGradientOp::Compute, scaleinvariantgradient.cc:117-195."""
    return run("ScaleInvariantGradient", [input], _sig_attrs(deltas, weights, epsilon))


def scale_invariant_gradient_grad(gradients, input, deltas=(1,), weights=(1.0,), epsilon=0.001):
    """ScaleInvariantGradientGradOp::Compute, scaleinvariantgradient.cc:294-404."""
    return run("ScaleInvariantGradientGrad", [gradients, input], _sig_attrs(deltas, weights, epsilon))


def depth_to_flow(depth, intrinsics, rotation, translation, rotation_format="angleaxis3", inverse_depth=False, normalize_flow=False):
    """DepthToFlowOp::Compute, depthtoflow.cc:211-313 (Eigen's rotation conversions come from oracle/ref_stub/eigen_stub.h)."""
    return run("DepthToFlow", [depth, intrinsics, rotation, translation],
               "rotation_format:s=%s;inverse_depth:b=%s;normalize_flow:b=%s" % (rotation_format, _b(inverse_depth), _b(normalize_flow)))


def replace_nonfinite(input, value=0.0):
    """ReplaceNonfiniteOp::Compute, replacenonfinite.cc:60-80."""
    return run("ReplaceNonfinite", [input], "value:f=%r" % float(value))


def replace_nonfinite_grad(gradients, input):
    """ReplaceNonfiniteGradOp::Compute, replacenonfinite.cc:123-150."""
    return run("ReplaceNonfiniteGrad", [gradients, input])


def depth_to_normals(depth, intrinsics, inverse_depth=False):
    """DepthToNormalsOp::Compute, depthtonormals.cc:117-238 (Matrix3::inverse, cross, normalize come from oracle/ref_stub/eigen_stub.h)."""
    return run("DepthToNormals", [depth, intrinsics], "inverse_depth:b=%s" % _b(inverse_depth))
