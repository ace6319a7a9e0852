"""CPU tests: the oracle against the reference's own known-answer outputs
(tests/golden/distance_kat.json, transcribed from test/expected/*.out) and against
what the reference's halfutils.c/bitutils.c return on fixed inputs
(tests/golden/ref_kernels.npz, recorded by tests/golden/make_ref_kernels.py)."""
import math
import os

import numpy as np
import pytest

import oracle as O
from tests.util import GOLDEN, f32_to_half_bits, half_bits_to_f32, load_golden, parse_vector

ELEM = {"vector": O.VECTOR, "halfvec": O.HALFVEC, "bit": O.BIT}
METRIC = {"l2_distance": O.L2, "inner_product": O.IP, "negative_inner_product": O.NEG_IP,
          "cosine_distance": O.COSINE, "l1_distance": O.L1, "hamming_distance": O.HAMMING,
          "jaccard_distance": O.JACCARD}

KAT = load_golden("distance_kat.json")["cases"]
REF_KERNELS = np.load(os.path.join(GOLDEN, "ref_kernels.npz"))


def _expect_float(text):
    if text == "NaN":
        return math.nan
    return float(text.replace("Infinity", "inf"))


@pytest.mark.parametrize("case", KAT, ids=[c["source"].split("/")[-1] for c in KAT])
def test_known_answer(case):
    elem = ELEM[case["type"]]
    fn = case["fn"]
    args = [parse_vector(a, elem) for a in case["args"]]
    if fn in METRIC:
        (a, da), (b, db) = args
        # varbit(n) casts in bit.out change the declared max length, not the value
        if case["error"]:
            assert da != db, case   # every distance error in these files is a dimension mismatch
            kind = "bit lengths" if elem == O.BIT else "vector dimensions" if elem == O.VECTOR else "halfvec dimensions"
            assert case["error"] == f"different {kind} {da} and {db}"
            return
        got = O.distance(elem, METRIC[fn], a, b, dim=da)
        want = _expect_float(case["expected"])
        if math.isnan(want):
            assert math.isnan(got)
        else:
            assert got == want, (case, got)
    elif fn in ("vector_norm", "l2_norm"):
        (a, _), = args
        got = O.norm(elem, a)
        if case["real"]:
            got = float(np.float32(got))
            assert np.float32(got) == np.float32(_expect_float(case["expected"]))
        elif case["expected"] is not None:
            assert got == _expect_float(case["expected"])
    elif fn == "l2_normalize":
        (a, _), = args
        if case["error"]:
            with pytest.raises(OverflowError):
                O.l2_normalize(elem, a)
            return
        got = O.l2_normalize(elem, a)
        want, _ = parse_vector(case["expected"], elem)
        if elem == O.HALFVEC:
            assert np.array_equal(got, want), (half_bits_to_f32(got), half_bits_to_f32(want))
        else:
            assert np.array_equal(got, want)
    elif fn == "binary_quantize":
        (a, d), = args
        got = O.binary_quantize(elem, a)
        want, _ = parse_vector(case["expected"], O.BIT)
        assert np.array_equal(got, want)
    else:
        pytest.fail(f"unhandled {fn}")


def test_kat_coverage():
    fns = {(c["type"], c["fn"]) for c in KAT}
    for t in ("vector", "halfvec"):
        for f in ("l2_distance", "inner_product", "cosine_distance", "l1_distance", "l2_normalize"):
            assert (t, f) in fns
    assert ("bit", "hamming_distance") in fns and ("bit", "jaccard_distance") in fns
    assert len(KAT) >= 100


def test_half_conversion_matches_reference_and_numpy():
    rng = np.random.default_rng(0)
    xs = np.concatenate([
        rng.standard_normal(2000).astype(np.float32) * 10,
        np.float32([0, -0.0, 1, -1, 65504, 65520, 65519.99, 1e-8, 5.96e-8, 2.98e-8, 2.9802322e-8, 6.1e-5, 6.0975552e-5,
                    1e5, -1e5, np.inf, -np.inf, 0.1, 0.33325195, 1.0009766, 1.00048828125, 1.0014648]),
        (rng.standard_normal(500) * 1e-6).astype(np.float32),
    ])
    L = O.lib()
    npbits = f32_to_half_bits(xs)
    for x, nb in zip(xs, npbits):
        ob = L.pgv_float_to_half(float(x))
        assert ob == int(nb), (x, ob, nb)
    G = REF_KERNELS
    for x, rb in zip(G["f2h_in"], G["f2h_out"]):
        assert L.pgv_float_to_half(float(x)) == int(rb), x
    # widening: all 65536 patterns
    allh = np.arange(65536, dtype=np.uint16)
    npf = half_bits_to_f32(allh)
    ref_h2f = dict(zip(G["h2f_in"].tolist(), G["h2f_out"].tolist()))
    for h in range(0, 65536, 7):
        f = L.pgv_half_to_float(h)
        if math.isnan(f):
            assert math.isnan(npf[h])
        else:
            assert f == npf[h]
            assert ref_h2f[h] == f


def test_restated_half_and_bit_kernels_match_reference_build():
    """The restatement vs the reference's own kernels on stored random inputs: bit kernels
    exactly; half kernels within fp32 reassociation noise of the fp64 truth."""
    G = REF_KERNELS
    for dim in (1, 3, 8, 9, 64, 100, 768, 1537):
        a, b = G[f"half_a_{dim}"], G[f"half_b_{dim}"]
        ref_l2sq, ref_ip, ref_l1, ref_cos = G[f"half_out_{dim}"]
        truth = O.distance(O.HALFVEC, O.L2_SQUARED, a, b, f64=True)
        for got in (ref_l2sq, O.distance(O.HALFVEC, O.L2_SQUARED, a, b)):
            assert abs(got - truth) <= 1e-5 * max(1.0, abs(truth))
        truth = O.distance(O.HALFVEC, O.IP, a, b, f64=True)
        scale = float(np.sum(np.abs(half_bits_to_f32(a) * half_bits_to_f32(b)))) + 1.0
        for got in (ref_ip, O.distance(O.HALFVEC, O.IP, a, b)):
            assert abs(got - truth) <= 1e-5 * scale
        truth = O.distance(O.HALFVEC, O.L1, a, b, f64=True)
        for got in (ref_l1, O.distance(O.HALFVEC, O.L1, a, b)):
            assert abs(got - truth) <= 1e-5 * max(1.0, truth)
        cos_ref = 1.0 - min(1.0, max(-1.0, ref_cos))
        assert abs(cos_ref - O.distance(O.HALFVEC, O.COSINE, a, b)) <= 1e-5
    for nbits in (0, 1, 7, 8, 52, 63, 64, 65, 513, 1024, 4099):
        a, b = G[f"bit_a_{nbits}"], G[f"bit_b_{nbits}"]
        assert int(G[f"bit_hamming_{nbits}"]) == O.distance(O.BIT, O.HAMMING, a, b, dim=nbits)
        assert float(G[f"bit_jaccard_{nbits}"]) == O.distance(O.BIT, O.JACCARD, a, b, dim=nbits)


def test_cross_type_equality_small_integers():
    """test/t/034_distance_functions.pl:36-52: halfvec distances print identically to vector
    distances on small-integer vectors, for all four metrics."""
    rng = np.random.default_rng(34)
    for _ in range(50):
        a = rng.integers(1, 10, size=5).astype(np.float32)
        b = rng.integers(1, 10, size=5).astype(np.float32)
        for m in (O.L2, O.IP, O.COSINE, O.L1):
            v = O.distance(O.VECTOR, m, a, b)
            h = O.distance(O.HALFVEC, m, f32_to_half_bits(a), f32_to_half_bits(b))
            assert v == h


def test_fp32_kernels_within_tolerance_of_truth():
    rng = np.random.default_rng(2)
    for dim in (3, 128, 1536, 2000):
        a = rng.standard_normal(dim).astype(np.float32)
        b = rng.standard_normal(dim).astype(np.float32)
        for m in (O.L2_SQUARED, O.L2, O.L1, O.COSINE):
            t = O.distance(O.VECTOR, m, a, b, f64=True)
            assert abs(O.distance(O.VECTOR, m, a, b) - t) <= 1e-5 * max(abs(t), 1e-30)
