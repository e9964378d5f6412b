"""CPU tests: the oracle against the reference's golden vectors and stored outputs of the reference's own C kernels.

These pin the oracle (task rule: an oracle must be checked against every golden vector / fixture the
reference's tests hold for the path, or against outputs of the reference itself).
"""
import hashlib
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def test_rope_table_matches_reference_golden(oracle):
    # TestCorrectness.TestRope (jlama-tests/.../model/TestCorrectness.java:93-115)
    g = json.load(open(os.path.join(HERE, "golden", "rope_testrope.json")))
    t = oracle.precompute_freqs_cis(128, 4096 * 2, 10000.0, 1.0)
    for i in range(64):
        assert abs(g["sin_position_1"][i] - t[i + 64, 1]) <= g["tolerance"]
        assert abs(g["sin_position_64"][i] - t[i + 64 * 64, 1]) <= g["tolerance"]


def test_float_types_roundtrip(oracle):
    # TestCorrectness.testFloatTypes (:138-145): bf16 round trip within 1e-2
    rng = np.random.default_rng(7)
    f = rng.uniform(-1, 1, 1000).astype(np.float32)
    back = oracle.bf16_to_f32(oracle.f32_to_bf16(f))
    assert np.abs(back - f).max() <= 0.01
    # RNE + NaN preservation (FloatConversions.java:35-61)
    x = np.array([1.0, 1.00390625, 1.01171875, np.nan, np.inf, -np.inf, 0.0], dtype=np.float32)
    b = oracle.f32_to_bf16(x)
    assert b[0] == 0x3F80 and b[1] == 0x3F80 and b[2] == 0x3F82  # ties to even
    assert b[3] == 0x7FC0 and b[4] == 0x7F80 and b[5] == 0xFF80 and b[6] == 0


# Outputs of the reference's own C kernels (jlama-native/src/main/c/simd/vector_simd.c) on the seeded inputs built below, stored by
# tests/golden/make_golden.py: "matches the reference" is checked on every machine, whether or not the reference's sources are at hand.
# The kernels ship a 512-bit and a 256-bit body of every kernel (vector_simd.c:465-468); "avx512" is the AVX-512 VNNI build, "avx2" the
# x86-64-v3 one.
REF_GOLDEN = os.path.join(HERE, "golden", "ref_kernels.npz")
GEMM_SHAPES = [(1, 128, 1024), (8, 64, 256), (32, 128, 1024), (7, 33, 512), (3, 16, 256)]
GEMM_8B_SHAPES = [(1, 320, 4096), (8, 320, 4096), (1, 320, 14336), (8, 160, 14336)]


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def gemm_inputs(M, N, K):
    # the reference's own distributions (TestOperations.java:94-109): A ~ U(-1,100), W ~ U(0,1)
    rng = np.random.default_rng(M * 1000 + N)
    return rng.uniform(-1, 100, (M, K)).astype(np.float32), rng.uniform(0, 1, (N, K)).astype(np.float32)


def gemm_8b_inputs(M, N, K):
    rng = np.random.default_rng(K + M)
    return rng.standard_normal((M, K)).astype(np.float32), (rng.standard_normal((N, K)) * 0.02).astype(np.float32)


def builds_inputs():
    rng = np.random.default_rng(77)
    return rng.standard_normal((4, 4096)).astype(np.float32), (rng.standard_normal((320, 4096)) * 0.02).astype(np.float32)


def dense_inputs():
    rng = np.random.default_rng(5)
    return rng.uniform(-1, 100, (5, 512)).astype(np.float32), rng.uniform(0, 1, (20, 512)).astype(np.float32)


def bf16_inputs():
    rng = np.random.default_rng(9)
    return rng.uniform(-1, 100, (4, 256)).astype(np.float32), rng.uniform(0, 1, (20, 256)).astype(np.float32)


def q4_products(oracle, a, w):
    """Q8 x Q4 and F32 x Q4 batch_dot of a and w through the reference's quantisers: the restatement, or the reference's kernels
    after oracle.use_reference_kernels(True)."""
    K, N = a.shape[1], w.shape[0]
    bq, bs = oracle.quantize_q4(w)
    aq, as_ = oracle.quantize_q8_act(a)
    B = oracle.OTensor(oracle.Q4, bq, bs)
    return oracle.batch_dot(oracle.OTensor(oracle.I8, aq, as_), B, 0, 0, K, 0, 0, N), oracle.batch_dot(oracle.f32(a), B, 0, 0, K, 0, 0, N)


@pytest.fixture(scope="module")
def ref_out():
    with np.load(REF_GOLDEN) as z:
        return {k: z[k] for k in z.files}


def reference(ref_out, key, *inputs):
    """The stored outputs of case `key`, after checking that this machine built the inputs they were computed on."""
    assert str(ref_out[key + ".inputs_sha256"]) == digest(*inputs), "%s: seeded inputs differ from those of %s" % (key, REF_GOLDEN)
    return lambda name: ref_out[key + "." + name]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_restatement_matches_reference_c_kernels(oracle, ref_out, M, N, K):
    a, w = gemm_inputs(M, N, K)
    ref = reference(ref_out, "gemm_%dx%dx%d" % (M, N, K), a, w)
    r_q8, r_f32 = q4_products(oracle, a, w)
    q_q8, q_f32 = ref("q8.avx512"), ref("f32.avx512")
    assert np.abs(r_q8 - q_q8).max() <= 2e-6 * np.abs(q_q8).max()
    assert np.abs(r_f32 - q_f32).max() <= 5e-6 * np.abs(q_f32).max()
    # and against the Naive control (get()*get() sequential), the reference tests' 1 % bar on the sum
    B = oracle.OTensor(oracle.Q4, *oracle.quantize_q4(w))
    naive = oracle.batch_dot(oracle.f32(a), B, 0, 0, K, 0, 0, N, naive=True)
    assert abs(naive.sum() - r_f32.sum()) <= 0.01 * abs(naive.sum())
    assert abs(naive.sum() - r_q8.sum()) <= 0.01 * abs(naive.sum())


@pytest.mark.parametrize("M,N,K", GEMM_8B_SHAPES)
def test_gemm_restatement_matches_reference_c_kernels_at_the_8b_reduction_lengths(oracle, ref_out, M, N, K):
    """The same pinning in the regime the benchmark runs in: K = 4096 (q/k/v/o, gate/up) and K = 14336 (down_proj) of Llama-3-8B, weights
    N(0, 0.02^2) through the reference's Q4 quantiser, activations N(0, 1) through its Q8 quantiser.  The two differ by summation order
    only; the float64 product of the dequantised operands bounds both."""
    a, w = gemm_8b_inputs(M, N, K)
    ref = reference(ref_out, "gemm8b_%dx%dx%d" % (M, N, K), a, w)
    r_q8, r_f32 = q4_products(oracle, a, w)
    q_q8, q_f32 = ref("q8.avx512"), ref("f32.avx512")
    assert not np.array_equal(r_f32, q_f32)  # two implementations really ran
    assert np.abs(r_q8 - q_q8).max() <= 3e-6 * np.abs(q_q8).max()
    assert np.abs(r_f32 - q_f32).max() <= 1e-5 * np.abs(q_f32).max()
    bq, bs = oracle.quantize_q4(w)
    aq, as_ = oracle.quantize_q8_act(a)
    wd = oracle.dequantize_q4(bq, bs).astype(np.float64)
    exact_f32 = a.astype(np.float64) @ wd.T
    exact_q8 = (aq.astype(np.float64).reshape(M, K // 32, 32) * as_.astype(np.float64)[:, :, None]).reshape(M, K) @ wd.T
    for got, exact in ((r_f32, exact_f32), (q_f32, exact_f32), (r_q8, exact_q8), (q_q8, exact_q8)):
        assert np.abs(got - exact).max() <= 1e-5 * np.abs(exact).max()


def test_both_reference_builds_bracket_the_restatement(oracle, ref_out):
    """The reference's 256-bit and 512-bit bodies sum in different orders, so they differ from each other by as much as either
    differs from the restatement -- the yardstick for every "matches the reference" bar."""
    a, w = builds_inputs()
    ref = reference(ref_out, "builds", a, w)
    port = q4_products(oracle, a, w)
    for i, kind, bar in ((0, "q8", 3e-6), (1, "f32", 1e-5)):
        out = {b: ref(kind + "." + b) for b in ("avx512", "avx2")}
        scale = np.abs(port[i]).max()
        d_builds = np.abs(out["avx512"] - out["avx2"]).max() / scale
        d_port = max(np.abs(out[b] - port[i]).max() / scale for b in out)
        assert d_builds <= bar and d_port <= bar
        assert d_builds > 0  # the two builds are not bit-identical: bit-exactness against "the reference" is not defined for these sums


def test_dense_f32_matches_reference_c_kernel(oracle, ref_out):
    a, w = dense_inputs()
    q = reference(ref_out, "dense_f32", a, w)("avx512")
    r = oracle.batch_dot(oracle.f32(a), oracle.f32(w), 0, 0, 512, 0, 0, 20)
    assert np.abs(r - q).max() <= 5e-6 * np.abs(q).max()


def test_f32_bf16_gemm_matches_reference_c_kernel(oracle, ref_out):
    # F32 x BF16 (vector_simd.h:38; PanamaTensorOperations.java:1466-1539): N a multiple of 5 because of the reference
    # splitter's corner-tile bug (DESIGN.md section 6).  The reference's gemm_bf16 (BF16 x BF16, vector_simd.h:34) returns
    # NaNs / wrong sums for the same call shape when driven directly through its C entry point, so BF16 x BF16 is pinned
    # only against the exact float64 product below.
    a, w = bf16_inputs()
    q1 = reference(ref_out, "f32_bf16", a, w)("avx512")
    wb = oracle.f32_to_bf16(w)
    ab = oracle.f32_to_bf16(a)
    exact = oracle.bf16_to_f32(ab).astype(np.float64) @ oracle.bf16_to_f32(wb).astype(np.float64).T
    r1 = oracle.batch_dot(oracle.f32(a), oracle.OTensor(oracle.BF16, wb), 0, 0, 256, 0, 0, 20)
    assert np.abs(r1 - q1).max() <= 5e-6 * np.abs(q1).max()
    r2 = oracle.batch_dot(oracle.OTensor(oracle.BF16, ab), oracle.OTensor(oracle.BF16, wb), 0, 0, 256, 0, 0, 20)
    assert np.abs(r2 - exact).max() <= 5e-6 * np.abs(exact).max()


def test_batch_dot_offsets_follow_panama_semantics(oracle):
    # result[i, j + rRowOffset] for j in [bRowOffset, bRowOffset+N) (PanamaTensorOperations.java:848)
    rng = np.random.default_rng(11)
    a = rng.standard_normal((2, 128)).astype(np.float32)
    w = rng.standard_normal((16, 128)).astype(np.float32)
    full = a[:, 32:96] @ w[:, 64:128].T
    r = np.zeros((2, 40), dtype=np.float32)
    oracle.batch_dot(oracle.f32(a), oracle.f32(w), 32, 64, 64, 20, 4, 8, result=r)
    assert np.allclose(r[:, 24:32], full[:, 4:12], rtol=1e-5, atol=1e-5)
    assert np.all(r[:, :24] == 0) and np.all(r[:, 32:] == 0)


def test_q4_block_format(oracle):
    # Q4ByteBufferTensor.java:66-120,179-197
    x = np.zeros((1, 32), dtype=np.float32)
    x[0, :] = np.linspace(-1.0, 0.9, 32)
    q, s = oracle.quantize_q4(x)
    assert s[0, 0] == np.float32(-1.0) / np.float32(-8.0)  # signed max / -8
    deq = oracle.dequantize_q4(q, s)
    assert deq[0, 0] == np.float32(-1.0)  # the max element is reproduced exactly (nibble 0 -> -8*scale)
    # byte j holds element j in the low nibble and element j+16 in the high nibble
    lo, hi = (q[0] & 0x0F).astype(int) - 8, (q[0] >> 4).astype(int) - 8
    assert np.allclose(lo * s[0, 0], deq[0, :16]) and np.allclose(hi * s[0, 0], deq[0, 16:])
    # all-zero block: scale 0 (Float.MIN_VALUE / -8 underflows), values 0
    q0, s0 = oracle.quantize_q4(np.zeros((1, 32), dtype=np.float32))
    assert s0[0, 0] == 0 and np.all(oracle.dequantize_q4(q0, s0) == 0)


def test_q8_activation_rounding_truncates_toward_zero(oracle):
    # PanamaTensorOperations.java:1705-1710: (byte)(x*id + 0.5f): positives round half up, negatives toward zero
    x = np.zeros((1, 32), dtype=np.float32)
    x[0, 0] = 127.0
    x[0, 1] = 2.5
    x[0, 2] = -2.5
    x[0, 3] = -2.6
    x[0, 4] = -0.4
    q, s = oracle.quantize_q8_act(x)
    assert s[0, 0] == np.float32(1.0)
    assert list(q[0, :5]) == [127, 3, -2, -2, 0]
    # weight-side quantiser uses Math.round instead (Q8ByteBufferTensor.java:87)
    qw, _ = oracle.quantize_q8_weights(x)
    assert list(qw[0, :5]) == [127, 3, -2, -3, 0]


def test_softmax_rmsnorm_silu_restatements(oracle):
    rng = np.random.default_rng(3)
    x = rng.standard_normal(50).astype(np.float32)
    y = oracle.softmax(x.copy().reshape(1, -1), 0, 50).ravel()
    e = np.exp(x.astype(np.float64) - x.max())
    assert np.allclose(y, e / e.sum(), rtol=2e-6)
    h = rng.standard_normal((3, 64)).astype(np.float32)
    w = (1 + 0.1 * rng.standard_normal((1, 64))).astype(np.float32)
    out = oracle.rmsnorm(h, oracle.f32(w), 1e-5)
    ref = h / np.sqrt((h.astype(np.float64) ** 2).mean(axis=1, keepdims=True) + 1e-5) * w
    assert np.allclose(out, ref, rtol=2e-6, atol=1e-6)
    s = oracle.silu(np.array([-3.0, 0.0, 2.0], dtype=np.float32))
    assert np.allclose(s, [-3 / (1 + np.exp(3)), 0, 2 / (1 + np.exp(-2))], rtol=1e-6)


def test_kv_page_solver_and_dctx(oracle):
    # SURVEY 8a a19: Llama-3-8B F32 -> 32 layers x 32 positions per 8 MiB page; 1B -> 16 x 128
    assert oracle.kv_page_solver(32, 8192, 1024) == (32, 32)
    assert oracle.kv_page_solver(16, 131072, 512) == (16, 128)
    # DistributedContext.java:75-98 for Llama-3-8B over 8 shards, shard 3
    d = oracle.dctx(4096, 4096, 14336, 128, 4, 32, 3, 8)
    assert (d.attentionSegmentStart, d.attentionSegmentLength) == (1536, 512)
    assert (d.kvSegmentStart, d.kvSegmentLength) == (384, 128)
    assert (d.hiddenSegmentStart, d.hiddenSegmentLength) == (5376, 1792)
    assert (d.headStart, d.headEnd, d.groupHeadStart, d.groupHeadEnd) == (12, 16, 3, 4)


def test_oracle_model_generate_is_deterministic_and_causal(oracle):
    from jlama_b200 import synth
    cfg = synth.get_config("tiny-mha")
    w = synth.make_weights(cfg)
    m = oracle.OracleLlama(cfg, w, act_q8=True)
    prompt = synth.random_prompt(cfg, 12)
    t1, l1 = m.generate(prompt, 6)
    t2, l2 = m.generate(prompt, 6)
    assert list(t1) == list(t2) and np.array_equal(l1, l2)
    # prefill in one chunk == prefill token by token (batchForward chunking must not change the result much)
    m.reset()
    h_batch = m.batch_forward(prompt, 0, max_batch=256)
    m.reset()
    for i, t in enumerate(prompt):
        h_tok = m.batch_forward([t], i, max_batch=256)
    assert np.allclose(h_batch, h_tok, rtol=1e-4, atol=1e-5)
    # tensor-parallel simulation (sum of column-shard partials) stays within float rounding
    m2 = oracle.OracleLlama(cfg, w, act_q8=True, tp=2)
    t3, l3 = m2.generate(prompt, 6)
    assert np.abs(l3 - l1).max() <= 1e-3 * np.abs(l1).max()
    m.close()
    m2.close()


def test_gpt2_restatement_is_self_consistent(oracle):
    """oracle.OracleGPT2 (GPT2Model.java:54-129 restated, incremental K/V) against a from-scratch float64 evaluation of the same network
    over the whole sequence (full causal attention matrix): pins the bookkeeping of the restatement (cache, splits of c_attn, biases,
    residual order); the reference holds no golden vectors for GPT-2 without a checkpoint (TestModels needs downloaded weights)."""
    from jlama_b200 import synth
    cfg = synth.get_gpt2_config("gpt2-tiny")
    w = synth.make_gpt2_weights(cfg)
    g = lambda n: np.asarray(w[n][1], dtype=np.float64)  # noqa: E731
    toks = synth.random_prompt(cfg, 11)
    E, nh, eps = cfg["E"], cfg["heads"], cfg["eps"]
    hs = E // nh

    def ln(x, wn, bn):
        mu = x.mean(-1, keepdims=True)
        var = (x * x).mean(-1, keepdims=True) - mu * mu
        return (x - mu) / np.sqrt(var + eps) * g(wn) + g(bn)

    x = g("wte.weight")[np.asarray(toks)] + g("wpe.weight")[:len(toks)]
    mask = np.triu(np.full((len(toks), len(toks)), -np.inf), 1)
    for i in range(cfg["layers"]):
        b = "h.%d." % i
        qkv = ln(x, b + "ln_1.weight", b + "ln_1.bias") @ g(b + "attn.c_attn.weight") + g(b + "attn.c_attn.bias")
        q, k, v = np.split(qkv, 3, axis=1)
        att = np.empty_like(q)
        for h in range(nh):
            sl = slice(h * hs, (h + 1) * hs)
            s = q[:, sl] @ k[:, sl].T / np.sqrt(hs) + mask
            p = np.exp(s - s.max(-1, keepdims=True))
            att[:, sl] = (p / p.sum(-1, keepdims=True)) @ v[:, sl]
        xb = att @ g(b + "attn.c_proj.weight") + g(b + "attn.c_proj.bias") + x
        hfc = ln(xb, b + "ln_2.weight", b + "ln_2.bias") @ g(b + "mlp.c_fc.weight") + g(b + "mlp.c_fc.bias")
        hfc = 0.5 * hfc * (1 + np.tanh(np.sqrt(2 / np.pi) * (hfc + 0.044715 * hfc ** 3)))
        x = hfc @ g(b + "mlp.c_proj.weight") + g(b + "mlp.c_proj.bias") + xb
    ref_logits = ln(x[-1:], "ln_f.weight", "ln_f.bias")[0] @ g("wte.weight").T
    om = oracle.OracleGPT2(cfg, w)
    ot, ol = om.generate(toks, 1)
    assert np.abs(ol[0] - ref_logits).max() <= 2e-5 * np.abs(ref_logits).max()
    assert ot[0] == int(np.argmax(ref_logits))
