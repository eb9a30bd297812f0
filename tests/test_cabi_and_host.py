"""CPU: the C-ABI library loads and exports every symbol include/demon_b200.h declares; the Python
mirrors validate shapes like the reference's shape functions without needing a GPU; the product never
falls back to a CPU implementation."""
import os
import re

import numpy as np
import pytest
import torch

from demon_b200 import _lib, build as dbuild

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    dbuild.build()
    return _lib.load()


def test_header_symbols_are_exported_and_bound(lib):
    header = open(os.path.join(ROOT, "include", "demon_b200.h")).read()
    declared = set(re.findall(r"\b(demon_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert lib.demon_version().decode().endswith("sm_100a")


def test_library_is_sm100a_only():
    """cuobjdump lists exactly one cubin architecture: sm_100a."""
    import subprocess
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.lib_path()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback():
    from demon_b200 import lmbspecialops as ops
    from demon_b200.networks_original import Session, BootstrapNet
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.median3x3_downsample(np.zeros((4, 4), np.float32))
    s = Session()
    s.load_weights({})
    with pytest.raises(RuntimeError, match="CUDA"):
        BootstrapNet(s).eval(np.zeros((1, 6, 192, 256), np.float32), np.zeros((1, 3, 48, 64), np.float32))


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "demon_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "liboracle" not in src, f


def test_shape_errors_match_reference_shape_functions():
    """test_FlowToDepth2.py:180-200: mismatching batch sizes -> ValueError 'Dimensions must be equal'."""
    from demon_b200 import lmbspecialops as ops
    batch = np.array([7, 7, 7, 5])
    for i in range(4):
        batch = np.roll(batch, 1)
        args = dict(flow=np.zeros((batch[0], 2, 6, 12), np.float32), rotation=np.zeros((batch[1], 3), np.float32),
                    translation=np.zeros((batch[2], 3), np.float32), intrinsics=np.zeros((batch[3], 4), np.float32))
        with pytest.raises(ValueError, match="Dimensions must be equal"):
            ops.flow_to_depth2(**args)
        with pytest.raises(ValueError, match="Dimensions must be equal"):
            ops.depth_to_flow(depth=np.zeros((batch[0], 1, 6, 12), np.float32), intrinsics=args["intrinsics"],
                              rotation=args["rotation"], translation=args["translation"])
    with pytest.raises(ValueError):   # C must be 2 (warp2d.cc:42-47)
        ops.warp2d(np.zeros((1, 3, 4, 5), np.float32), np.zeros((1, 3, 4, 5), np.float32))
    with pytest.raises(ValueError):   # H, W must agree (warp2d.cc:50-60)
        ops.warp2d(np.zeros((1, 3, 4, 5), np.float32), np.zeros((1, 2, 4, 6), np.float32))
    with pytest.raises(ValueError):   # intrinsics last dim 4 (depthtoflow.cc:58-62)
        ops.depth_to_flow(np.zeros((1, 1, 4, 5), np.float32), np.zeros((1, 3)), np.zeros((1, 3)), np.zeros((1, 3)))
    with pytest.raises(ValueError):   # quaternion has 4 elements (depthtoflow.cc:72-75)
        ops.depth_to_flow(np.zeros((1, 1, 4, 5), np.float32), np.zeros((1, 4)), np.zeros((1, 3)), np.zeros((1, 3)),
                          rotation_format="quaternion")
    with pytest.raises(ValueError, match="deltas and weights"):   # scaleinvariantgradient.cc:115-117
        ops.scale_invariant_gradient(np.zeros((4, 4), np.float32), deltas=[1, 2], weights=[1.0])
    with pytest.warns(DeprecationWarning):   # the deprecated twin warns, then validates like flow_to_depth2
        with pytest.raises(ValueError, match="Dimensions must be equal"):
            ops.flow_to_depth(np.zeros((1, 2, 4, 5), np.float32), np.zeros((2, 4), np.float32), np.zeros((1, 3), np.float32),
                              np.zeros((1, 3), np.float32))


def test_network_argument_validation():
    from demon_b200.networks_original import Session, BootstrapNet, RefinementNet
    with pytest.raises(ValueError):
        BootstrapNet(Session(), data_format="NCHW")
    with pytest.raises(ValueError):
        Session(precision="fp8")
    with pytest.raises(ValueError):
        RefinementNet(Session(), image_size=(190, 256))
    with pytest.raises(RuntimeError, match="load_weights"):
        Session().net(1)
