"""Generates tests/golden/reference_ops.json: the digests (oracle.ref.output_digest: dtype, shape, SHA-256 of the bits)
of the outputs of the reference's OWN op kernels (oracle/_ref/libref_ops.so, built by oracle/ref.py from the
reference's lmbspecialops/src/*.cc against oracle/ref_stub/) on every case that tests/test_oracle_ref.py and
tests/test_gpu_training_ops.py compare with.  The cases come from the test modules themselves (their
`reference_cases()`), so inputs are defined once.  A digest holds an output bit for bit in a few bytes (the largest
output is 1.1 MB).  Needs the reference source tree:
    python tests/golden/make_reference_ops_golden.py
"""
import importlib.util
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_ops.json")
TEST_MODULES = ("test_oracle_ref", "test_gpu_training_ops")


def main():
    sys.path.insert(0, ROOT)
    from oracle import ref
    if ref.build() is None:
        raise SystemExit("the reference op sources are not present (oracle/ref.py REF_SRC)")
    out = {}
    for name in TEST_MODULES:
        spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tests", name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        for key, op, args in mod.reference_cases():
            assert key not in out, key
            out[key] = ref.output_digest(getattr(ref, op)(*args))
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", OUT, len(out), "digests")


if __name__ == "__main__":
    main()
