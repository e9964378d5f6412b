"""Regenerates tests/golden/ from the reference (a checkout of tjake/Jlama); the tests only read the committed files.

  python tests/golden/make_golden.py /path/to/Jlama

rope_testrope.json : the two 64-value expected sin arrays of TestCorrectness.TestRope
                     (jlama-tests/src/test/java/com/github/tjake/jlama/model/TestCorrectness.java:93-115),
                     the only golden vectors the reference holds for the hot path (SURVEY 8c).
ref_kernels.npz    : outputs of the reference's own C kernels (jlama-native/src/main/c/simd/vector_simd.c, built into oracle/_ref/
                     by oracle/Makefile) on the seeded inputs of tests/test_oracle.py, with a sha256 of those inputs per case.
                     Needs a CPU that runs both builds (AVX-512 VNNI and AVX2).
"""
import json
import os
import re
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TEST_CORRECTNESS = "jlama-tests/src/test/java/com/github/tjake/jlama/model/TestCorrectness.java"


def rope(reference):
    src = open(os.path.join(reference, TEST_CORRECTNESS)).read()
    blk = src[src.index("public void TestRope()"):src.index("public void testRope2()")]
    arrs = re.findall(r"new double\[\] \{(.*?)\};", blk, flags=re.S)
    vals = [[float(v) for v in a.replace("\n", " ").split(",") if v.strip()] for a in arrs]
    assert len(vals) == 2 and all(len(v) == 64 for v in vals)
    json.dump({"source": TEST_CORRECTNESS + ":93-115 (TestRope)",
               "call": "VectorMath.precomputeFreqsCis(128, 8192, 10000.0, 1.0)", "tolerance": 1e-4,
               "sin_position_1": vals[0], "sin_position_64": vals[1]},
              open(os.path.join(HERE, "rope_testrope.json"), "w"), indent=1)


def ref_kernels(reference):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + os.path.abspath(reference)])
    sys.path[:0] = [ROOT, os.path.dirname(HERE)]
    from oracle import oracle as o
    import test_oracle as t
    out = {}

    def use(build):
        assert o.load_reference_kernels(build) is not None, "this CPU cannot run the %s build" % build

    def products(key, build, a, w):
        use(build)
        o.use_reference_kernels(True)
        out[key + ".q8." + build], out[key + ".f32." + build] = t.q4_products(o, a, w)
        o.use_reference_kernels(False)
        out[key + ".inputs_sha256"] = np.array(t.digest(a, w))

    for shape in t.GEMM_SHAPES:
        products("gemm_%dx%dx%d" % shape, "avx512", *t.gemm_inputs(*shape))
    for shape in t.GEMM_8B_SHAPES:
        products("gemm8b_%dx%dx%d" % shape, "avx512", *t.gemm_8b_inputs(*shape))
    for build in ("avx512", "avx2"):
        products("builds", build, *t.builds_inputs())
    use("avx512")
    a, w = t.dense_inputs()
    out["dense_f32.avx512"], out["dense_f32.inputs_sha256"] = o.ref_gemm_f32(a, w, 0, w.shape[0]), np.array(t.digest(a, w))
    a, w = t.bf16_inputs()
    out["f32_bf16.avx512"] = o.ref_gemm_f32_bf16(a, o.f32_to_bf16(w), 0, w.shape[0])
    out["f32_bf16.inputs_sha256"] = np.array(t.digest(a, w))
    np.savez_compressed(os.path.join(HERE, "ref_kernels.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    rope(sys.argv[1])
    ref_kernels(sys.argv[1])
