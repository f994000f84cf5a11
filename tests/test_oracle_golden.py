"""Pins the CPU oracle (oracle/ronk_oracle.c) against every known-answer vector the reference's
own tests hold for the hot path (tests/golden/reference_kats.json, transcribed with file:line) and
against the independent pure-Python Goldilocks vectors (tests/golden/goldilocks_vectors.json).
CPU only."""
import os

import numpy as np
import pytest

import oracle
from conftest import pt

GL = oracle.GOLDILOCKS


def test_field_kats(kats):
    f = kats["field"]
    for p, a, b, r in f["add"]:
        assert oracle.add(p, a, b) == r
    for p, a, b, r in f["sub"]:
        assert oracle.sub(p, a, b) == r
    for p, a, b, r in f["mul"]:
        assert oracle.mul(p, a, b) == r
    for p, a, e, r in f["pow"]:
        assert oracle.pow_(p, a, e) == r
        assert oracle.pow_literal(p, a, e) == r  # delta D2 changes no value
    for p, a, r in f["inverse"]:
        assert oracle.inverse(p, a) == r
    for p in f["inverse_of_zero_panics"]:
        with pytest.raises(oracle.OraclePanic):
            oracle.inverse(p, 0)
    for p, a, r in f["halve"]:
        assert oracle.div(p, a, 2) == r
    for p, g in f["generator"].items():
        assert oracle.generator(int(p)) == g
    for p, n in f["no_root_of_unity"]:
        with pytest.raises(oracle.OraclePanic):
            oracle.root_of_unity(p, n)
    for n in f["non_prime_modulus_panics"]:
        assert oracle.lib().orc_is_prime(n) == 0
    assert oracle.lib().orc_is_prime(101) == 1 and oracle.lib().orc_is_prime(17) == 1


@pytest.mark.parametrize("p", [17, 101])
def test_field_exhaustive_laws(p):
    """prime/mod.rs:297-374: generator has order P-1; identities; inverse∘inverse; negation."""
    g = oracle.generator(p)
    seen, x = set(), 1
    for _ in range(p - 1):
        x = oracle.mul(p, x, g)
        seen.add(x)
    assert len(seen) == p - 1
    for a in range(p):
        assert oracle.add(p, a, 0) == a and oracle.mul(p, a, 1) == a and oracle.mul(p, a, 0) == 0
        assert oracle.add(p, a, oracle.neg(p, a)) == 0
        if a:
            assert oracle.inverse(p, oracle.inverse(p, a)) == a
            assert oracle.mul(p, a, oracle.inverse(p, a)) == 1


def test_polynomial_kats(kats):
    k = kats["polynomial"]
    p, a, b = k["p"], k["a"], k["b"]
    a5 = a + [0]
    assert list(oracle.poly_add(p, b, a)) == k["b_plus_a"]
    assert list(oracle.poly_sub(p, a5, b)) == k["a5_minus_b"]
    assert list(oracle.poly_sub(p, b, a5)) == k["b_minus_a5"]
    assert list(oracle.poly_neg(p, a)) == k["neg_a"]
    assert list(oracle.poly_mul(p, a, b)) == k["a_times_b"]
    assert list(oracle.poly_mul(p, k["c"], k["d"])) == k["c_times_d"]
    q, r = oracle.poly_divrem(p, a, b)
    assert list(q) == k["a_div_b"] and list(r) == k["a_rem_b"]
    q, r = oracle.poly_divrem(p, b, a)
    assert list(q) == k["b_div_a"] and list(r) == k["b_rem_a"]
    q, r = oracle.poly_divrem(p, [1, 2, 1], [1, 1])
    assert list(q) == k["p121_div_11"] and list(r) == k["p121_rem_11"]
    assert oracle.poly_eval(p, a, 2) == k["eval_a_at_2"]
    e = k["eval_103_at_0"]
    assert oracle.poly_eval(p, e["coeffs"], e["x"]) == e["y"]
    assert list(oracle.dft(p, a)) == k["dft_a"]
    assert list(oracle.fft(p, a)) == k["fft_a"]
    assert list(oracle.ntt_fast(p, a)) == k["fft_a"]
    assert list(oracle.ifft(p, oracle.fft(p, a))) == a
    assert oracle.lagrange_eval(p, oracle.dft(p, a), 2) == k["lagrange_eval_dft_a_at_2"]
    assert oracle.poly_degree(a) == k["degree_a"] and oracle.poly_leading(a) == k["leading_a"]
    assert list(oracle.poly_pow_mult(p, a, 2, 5)) == k["pow_mult_a_2_5"]
    with pytest.raises(oracle.OraclePanic):
        oracle.dft(p, k["dft_3_terms_panics"])
    c1 = kats["config1_extra"]
    assert list(oracle.poly_mul(c1["p"], c1["a"], c1["b"])) == c1["out"]


def test_gf101_2_kats(kats):
    g = kats["gf101_2"]
    for a, b, r in g["add"]:
        assert oracle.gf_add(a, b) == tuple(r)
    for a, r in g["neg"]:
        assert oracle.gf_neg(a) == tuple(r)
    for a, b, r in g["sub"]:
        assert oracle.gf_sub(a, b) == tuple(r)
    for a, b, r in g["mul"]:
        assert oracle.gf_mul(a, b) == tuple(r)
    # gf_101_2.rs:201-221 style law: a * a^-1 == 1 over the whole field
    for a0 in range(0, 101, 7):
        for a1 in range(0, 101, 5):
            if a0 or a1:
                assert oracle.gf_mul((a0, a1), oracle.gf_inv((a0, a1))) == (1, 0)
    # direct formula (a0b0 - 2a1b1, a0b1 + a1b0) equals the reference's poly-mul-then-% route
    rng = np.random.default_rng(1)
    for _ in range(200):
        a0, a1, b0, b1 = (int(v) for v in rng.integers(0, 101, 4))
        assert oracle.gf_mul((a0, a1), (b0, b1)) == ((a0 * b0 - 2 * a1 * b1) % 101, (a0 * b1 + a1 * b0) % 101)


def test_curve_kats(kats):
    c = kats["curve"]
    G1, G2 = bytes(c["G1"]), bytes(c["G2"])
    assert oracle.on_curve(G1) and oracle.on_curve(G2) and not oracle.on_curve(bytes(c["off_curve"]))
    for k, v in c["multiples_of_G1"].items():
        assert oracle.point_smul(G1, int(k)) == bytes(v)
    assert oracle.point_double(G1) == bytes(c["multiples_of_G1"]["2"])
    assert oracle.point_add(G1, oracle.point_double(G1)) == bytes(c["multiples_of_G1"]["3"])
    for a, b in c["negatives"]:
        assert oracle.point_neg(bytes(a)) == bytes(b)
    assert oracle.point_double(G2) == bytes(c["two_G2"])
    assert oracle.point_add(G1, oracle.INF) == G1 and oracle.point_add(oracle.INF, G1) == G1
    assert oracle.point_add(G1, oracle.point_neg(G1)) == oracle.INF
    # order 17 (pluto_curve.rs:128-137; kzg/tests.rs:240-252): 17·G = ∞ via repeated addition
    for G in (G1, G2):
        acc = G
        for _ in range(16):
            acc = oracle.point_add(acc, G)
        assert acc == oracle.INF


def test_kzg_kats(kats):
    k = kats["kzg"]
    g1, g2 = oracle.setup()
    assert g1 == [bytes(v) for v in k["g1srs"]] and g2 == [bytes(v) for v in k["g2srs"]]
    for c in k["commit"]:
        assert oracle.commit(c["coeffs"], g1) == pt(c["out"])
        assert oracle.commit(c["coeffs"], g1, fast=True) == pt(c["out"])
    acc = oracle.INF
    for i, s in k["srs_open"]["terms"]:
        acc = oracle.point_add(acc, oracle.point_smul(g1[i], s))
    assert acc == bytes(k["srs_open"]["out"])
    for o in k["open"]:
        assert oracle.open_(o["coeffs"], o["z"], g1) == bytes(o["out"])
    with pytest.raises(oracle.OraclePanic):  # kzg/setup.rs:53 assert
        oracle.commit([1] * 8, g1)


def test_reed_solomon_decode_kats(kats):
    """decoding / decoding_longer_message (src/codes/reed_solomon.rs:177-219): encode to N = 7, decode the
    first K coordinates with the literal combination formula (:55-107)."""
    r = kats["reed_solomon_decode"]
    for msg in r["messages"]:
        xs, ys = oracle.rs_encode(r["p"], msg, r["n"])
        assert list(oracle.rs_decode(r["p"], xs, ys, len(msg))) == msg
    # on a full set of roots of unity the interpolant is the inverse transform
    msg = oracle.splitmix(GL, 3, 8)
    xs, ys = oracle.rs_encode(GL, msg, 8)
    assert np.array_equal(oracle.rs_decode(GL, xs, ys, 8), msg) and np.array_equal(oracle.ifft(GL, ys), msg)
    with pytest.raises(oracle.OraclePanic):
        oracle.rs_decode(127, [1, 1, 2], [3, 4, 5], 3)   # repeated x: division by zero


def test_reed_solomon_kat(kats):
    r = kats["reed_solomon"]
    xs, ys = oracle.rs_encode(r["p"], r["msg"], r["n"])
    assert list(xs) == r["x"] and list(ys) == r["y"]


def test_commit_fast_matches_literal():
    rng = np.random.default_rng(7)
    G1, G2 = bytes([1, 0, 2, 0]), bytes([36, 0, 0, 31])
    pts = []
    for _ in range(300):
        k, l = (int(v) for v in rng.integers(0, 17, 2))
        pts.append(oracle.point_add(oracle.point_smul(G1, k), oracle.point_smul(G2, l)))
    sc = rng.integers(0, 17, 300).astype(np.uint8)
    assert oracle.commit(sc, pts) == oracle.commit(sc, pts, fast=True)


# ---- 64-bit (Goldilocks): pinned by the independent pure-Python vectors -----------------------
def _summary(x):
    n = len(x)
    idx = np.arange(1, n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        return {
            "first": int(x[0]), "second": int(x[1]), "last": int(x[-1]),
            "sum_mod_2_64": int(np.sum(x, dtype=np.uint64)),
            "weighted_sum_mod_2_64": int(np.sum(x * idx, dtype=np.uint64)),
            "xor": int(np.bitwise_xor.reduce(x)),
        }


def test_goldilocks_roots_and_small(gold64):
    for k, w in gold64["roots"].items():
        assert oracle.root_of_unity(GL, 1 << int(k)) == w
    for k, v in gold64["inv_n"].items():
        assert oracle.inverse(GL, 1 << int(k)) == v
    assert list(oracle.fft(GL, list(range(1, 9)))) == gold64["ntt8_1to8"]
    assert list(oracle.splitmix(GL, 42, 3)) == gold64["splitmix42_first3"]
    a = oracle.splitmix(GL, 42, 1024)
    assert list(oracle.fft(GL, a)) == gold64["ntt_2_10_full"]
    assert list(oracle.ntt_fast(GL, a)) == gold64["ntt_2_10_full"]
    assert list(oracle.dft(GL, a[:64])) == list(oracle.fft(GL, a[:64]))


@pytest.mark.parametrize("lg", [16, 20])
def test_goldilocks_ntt_summaries(gold64, lg):
    n = 1 << lg
    a = oracle.splitmix(GL, 42, n)
    X = oracle.fft(GL, a)  # faithful recursive
    g = gold64["ntt_2_%d" % lg]
    s = _summary(X)
    for key in s:
        assert s[key] == g[key], key
    for k, v in g["horner_checks"].items():
        assert int(X[int(k)]) == v
    assert np.array_equal(oracle.ntt_fast(GL, a), X)
    assert np.array_equal(oracle.ifft(GL, X), a)


def test_goldilocks_conv_and_mul(gold64):
    n = 1 << 16
    a, b = oracle.splitmix(GL, 42, n), oracle.splitmix(GL, 43, n)
    X, Y = oracle.ntt_fast(GL, a), oracle.ntt_fast(GL, b)
    Z = np.array([oracle.mul(GL, int(x), int(y)) for x, y in zip(X, Y)], dtype=np.uint64)
    c = oracle.ntt_fast(GL, Z, inverse=True)
    g = gold64["cyclic_conv_2_16_seed42_seed43"]
    s = _summary(c)
    for key in s:
        assert s[key] == g[key], key
    a3, b3 = oracle.splitmix(GL, 42, 300), oracle.splitmix(GL, 43, 300)
    assert list(oracle.poly_mul(GL, a3, b3)) == gold64["poly_mul_300x300_seed42_seed43"]
    e = gold64["eval_300_seed42_at_seed43_0"]
    assert oracle.poly_eval(GL, a3, e["x"]) == e["y"]


def test_next_rows_against_independent_vectors():
    """SURVEY §8f rows over the 64-bit field, pinned like the transforms: the C oracle against vectors from an
    independent pure-Python generator (tests/golden/gen_next_rows.py → next_rows_vectors.json)."""
    import json
    from gpu_util import summary
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "next_rows_vectors.json")))
    d = g["div_linear_5000_seed77"]
    q, r = oracle.poly_divrem(GL, oracle.splitmix(GL, 77, 5000), [d["b0"], d["b1"]])
    s = summary(q)
    assert all(s[k] == d["quotient"][k] for k in s) and int(r[0]) == d["remainder"] and not r[1:].any()
    d = g["divrem_40_by_5_seed1_seed2"]
    q, r = oracle.poly_divrem(GL, oracle.splitmix(GL, 1, 40), oracle.splitmix(GL, 2, 5))
    assert [int(v) for v in q] == d["q"] and [int(v) for v in r] == d["r"]
    d = g["rs_msg5_n8_seed3"]
    xs, ys = oracle.rs_encode(GL, d["msg"], 8)
    assert [int(v) for v in xs] == d["xs"] and [int(v) for v in ys] == d["ys"]
    assert [int(v) for v in oracle.rs_decode(GL, xs, ys, 5)] == d["msg"]
    d = g["interpolate_12_seed71_seed72"]
    assert [int(v) for v in oracle.rs_decode(GL, d["xs"], d["ys"], 12)] == d["coeffs"]


def test_kat_provenance_is_mechanical():
    """tests/golden/extract_reference_kats.py checks every vector of reference_kats.json against the reference's
    rstest tables and the cited Rust source, as parsed and located there and stored in reference_kat_sources.json."""
    import json
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "extract_reference_kats.py")
    out = subprocess.run([sys.executable, script], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout[-2000:]
    assert json.loads(out.stdout)["located"] >= 114


def test_extended_curve_has_102_squared_points_and_exponent_102():
    """What the histogram form of kzg::commit (msm.cu) relies on: E(F_101²): y² = x³ + 3 has 102² points (with
    Infinity) and every point is killed by 102, so Σ s_i·P_i = Σ_P (c_P mod 102)·P.  Enumerated with the oracle's
    own on-curve predicate and addition law (curve/mod.rs:130-139, :178-213)."""
    q = 101

    def gmul(a, b):
        return ((a[0] * b[0] - 2 * a[1] * b[1]) % q, (a[0] * b[1] + a[1] * b[0]) % q)

    roots = {}
    for y0 in range(q):
        for y1 in range(q):
            roots.setdefault(gmul((y0, y1), (y0, y1)), []).append((y0, y1))
    pts = []
    for x0 in range(q):
        for x1 in range(q):
            x = (x0, x1)
            r = gmul(gmul(x, x), x)
            for y in roots.get(((r[0] + 3) % q, r[1]), []):
                pts.append(bytes([x0, x1, y[0], y[1]]))
    assert len(pts) + 1 == 102 * 102
    rng = np.random.default_rng(1)
    sample = [pts[i] for i in rng.choice(len(pts), 400, replace=False)] + pts[:50] + pts[-50:]

    def smul(p, k):
        acc = oracle.INF
        for bit in bin(k)[2:]:
            acc = oracle.point_add(acc, acc)
            if bit == "1":
                acc = oracle.point_add(acc, p)
        return acc

    for p in sample:
        assert oracle.on_curve(p) and smul(p, 102) == oracle.INF
