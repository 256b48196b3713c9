"""The adversarial NN inputs (tests/nn_adversarial.py) really are adversarial, and the two CPU oracles agree on them.
No GPU: this shows what tests/test_gpu_nn_adversarial.py feeds the kernels.

For every generator and model variant:
  - the FP64 oracle's relative gap (second - first) / first falls into the buckets where the kernels' FP32 error bands
    decide (exact ties, below 1e-12, ..., below 1e-5) often enough -- the minimum counts are shares of the queries;
  - a naive FP32 decision (oracle-free, nn_adversarial.naive_fp32) picks the wrong point for a stated share of them;
  - oracle.nn_kdtree (the CPU baseline, with its 1e-9 re-decision band) equals oracle.nn_brute bit for bit."""
import numpy as np
import pytest

import nn_adversarial as A
import oracle

# generator -> minimum share of the queries per gap bucket [exact, (0,1e-12), [1e-12,1e-9), [1e-9,1e-7), [1e-7,1e-6), [1e-6,1e-5)]
# (None: no requirement), minimum share a naive FP32 decision gets wrong (float32 model, float64 model)
BUCKETS = {
    "bisector": ([None, None, 0.05, 0.10, 0.07, 0.06], 0.15, 0.35),
    "ties": ([1.0, None, None, None, None, None], 0.01, 0.35),
    "far": ([None, 0.20, 0.15, 0.10, 0.06, 0.05], 0.25, 0.30),
    "crowd": ([None, None, None, None, None, 0.04], 0.0, 0.20),
    "huge": ([0.6, 0.1, 0.05, 0.02, None, None], 0.8, 0.8),
}
# below 1e-9 together (exact ties and FP64-rounding-level gaps): the bucket split depends on the offset's FP64 resolution
BELOW_1E9 = dict(bisector=0.25, ties=1.0, far=0.25, crowd=0.0, huge=0.8)


@pytest.mark.parametrize("v", A.VARIANTS, ids=[A.variant_id(v) for v in A.VARIANTS])
@pytest.mark.parametrize("name", list(A.GENERATORS))
def test_inputs_are_adversarial(name, v):
    model, q = A.generate(name, v, **({"nq": 800} if name == "huge" else {}))
    oi, od = oracle.nn_brute(model, q)
    gap = A.gaps(model, q, oi, od)
    counts = A.gap_buckets(gap)
    mins, naive32, naive64 = BUCKETS[name]
    nq = q.shape[0]
    for b, (c, lo) in enumerate(zip(counts, mins)):
        if lo is not None:
            assert c >= lo * nq, "bucket %d: %d of %d queries (want >= %g): %s" % (b, c, nq, lo, counts)
    assert sum(counts[:3]) >= BELOW_1E9[name] * nq, counts
    # a variant whose coordinates round the crowd apart in FP32 already (float32 at offset 1e5) is exempt
    want = naive32 if v[0] == np.float32 else naive64
    if name == "crowd" and v[0] == np.float32 and v[1] >= 1e5:
        want = 0.0
    wrong = np.mean(A.naive_fp32(model, q) != oi)
    assert wrong >= want, "naive FP32 wrong on %.3f of the queries (want >= %g)" % (wrong, want)
    ki, kd = oracle.nn_kdtree(model, q)
    assert np.array_equal(ki, oi) and np.array_equal(kd, od), "nn_kdtree differs from nn_brute on %d queries" % int(np.sum(ki != oi))


def test_exact_ties_are_exact_and_fp32_inexact():
    """the tie generator's pairs tie exactly in FP64, yet their float32 roundings differ (float64 models), and the smaller
    original index is the FP32 winner for only part of them"""
    model, q = A.ties(5, np.float64, 1e3, 1.0, nq=1000)
    oi, od = oracle.nn_brute(model, q)
    sec = oracle.nn.nn_second(model, q, oi)
    assert np.array_equal(sec, od)
    m32 = model.astype(np.float32).astype(np.float64)
    assert np.mean(np.any(m32 != model, axis=1)) > 0.99
    naive = A.naive_fp32(model, q)
    assert 0.2 < np.mean(naive != oi) < 0.8
