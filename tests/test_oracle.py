"""Pins the oracle (oracle/seal_oracle.c): reference in-source KATs, committed golden vectors generated from the real
reference, and -- where oracle/_ref/libsealref.so is present -- live comparison with the reference itself."""
import numpy as np
import pytest

import oracle as O
import refseal as R
from common import golden, rand_ct

Q_KAT = 0xFFFFFFFFFFC0001


def test_kat_ntt_root_powers():
    # native/tests/seal/util/ntt.cpp:53-73
    oc = O.Oracle(O.CKKS, 2, [Q_KAT])
    root, rp, irp, _ = oc.ntt_tables(0)
    assert rp[0] == 1 and rp[1] == 288794978602139552
    assert (int(rp[1]) * int(irp[1])) % Q_KAT == 1
    oc = O.Oracle(O.CKKS, 4, [Q_KAT])
    _, rp, _, _ = oc.ntt_tables(0)
    assert list(map(int, rp)) == [1, 288794978602139552, 178930308976060547, 748001537669050592]


def test_kat_ntt_values():
    # native/tests/seal/util/ntt.cpp:75-100
    oc = O.Oracle(O.CKKS, 2, [Q_KAT])
    assert list(oc.ntt_row(0, np.array([0, 0], dtype=np.uint64))) == [0, 0]
    assert list(oc.ntt_row(0, np.array([1, 0], dtype=np.uint64))) == [1, 1]
    assert list(map(int, oc.ntt_row(0, np.array([1, 1], dtype=np.uint64)))) == [288794978602139553, 864126526004445282]


def test_kat_ntt_roundtrip():
    # native/tests/seal/util/ntt.cpp:103-133 (n = 8)
    oc = O.Oracle(O.CKKS, 8, [Q_KAT])
    rng = np.random.default_rng(0x5EA1)
    x = rng.integers(0, Q_KAT, 8, dtype=np.uint64)
    assert (oc.intt_row(0, oc.ntt_row(0, x)) == x).all()
    assert (oc.intt_row(0, np.zeros(8, dtype=np.uint64)) == 0).all()


def test_kat_galois():
    # native/tests/seal/util/galois.cpp:86-120 (n=8, q=17, g=3)
    x = np.arange(8, dtype=np.uint64)
    assert list(O.galois_coeff_row(8, 17, 3, x)) == [0, 14, 6, 1, 13, 7, 2, 12]
    assert list(O.galois_ntt_row(8, 3, x)) == [4, 5, 7, 6, 1, 0, 2, 3]


def test_kat_galois_elts():
    # native/tests/seal/util/galois.cpp:28-69 (EltFromStep for n = 8: generator 3 mod 16)
    assert O.galois_elt_from_step(8, 0) == 15
    assert O.galois_elt_from_step(8, 1) == 3
    assert O.galois_elt_from_step(8, -3) == 3
    assert O.galois_elt_from_step(8, 2) == 9
    assert O.galois_elt_from_step(8, -2) == 9
    assert O.galois_elt_from_step(8, 3) == 11
    assert O.galois_elt_from_step(8, -1) == 11


def test_default_moduli_known_values():
    # util/globals.cpp:43 BFVDefault(4096) = {0xffffee001, 0xffffc4001, 0x1ffffe0001}; CoeffModulus::Create hands equal-size
    # primes out smallest-first (modulus.cpp:175-181), so Create(4096,{36,36,37}) is the same set in ascending order
    assert O.coeff_modulus_create(4096, [36, 36, 37]) == [0xFFFFC4001, 0xFFFFEE001, 0x1FFFFE0001]
    assert all(O.lib().orc_is_prime(p) and p % 8192 == 1 for p in (0xFFFFEE001, 0xFFFFC4001, 0x1FFFFE0001))


@pytest.mark.parametrize("name", ["ckks_n128", "bfv_n128", "ckks_n1024", "bgv_n128"])
def test_oracle_vs_golden(name):
    g = golden(name)
    scheme, n, mods, t = int(g["scheme"]), int(g["n"]), [int(x) for x in g["moduli"]], int(g["t"])
    k = len(mods)
    oc = O.Oracle(scheme, n, mods, t)
    for i in range(k):
        assert oc.ntt_tables(i)[0] == int(g["roots"][i])
    key = g["relin_key"]
    for L in range(k - 1, 0, -1):
        a, b = g[f"L{L}_a"], g[f"L{L}_b"]
        assert (oc.ntt_forward(L, a) == g[f"L{L}_ntt_fwd_a"]).all()
        assert (oc.ntt_inverse(L, a) == g[f"L{L}_ntt_inv_a"]).all()
        m = oc.multiply(L, a, b)
        assert (m == g[f"L{L}_mul"]).all()
        assert (oc.relinearize(L, m, key) == g[f"L{L}_relin"]).all()
        if L > 1:
            ms = oc.rescale(L, a) if scheme == O.CKKS else (oc.bfv_mod_switch(L, a) if scheme == O.BFV else oc.bgv_mod_switch(L, a))
            assert (ms == g[f"L{L}_modswitch_a"]).all()
        for e in g["galois_elts"]:
            e = int(e)
            assert (oc.apply_galois(L, a, e, g[f"galois_key_{e}"]) == g[f"L{L}_galois_{e}"]).all()
        if scheme == O.BFV:
            assert oc.base_bsk(L) == [int(x) for x in g[f"L{L}_bsk"]]


needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libsealref.so not built")


@needs_ref
def test_oracle_vs_live_reference_ckks():
    # non-descending chain (50/40/45/60 bits) exercises both conditional-reduction branches (evaluator.cpp:2690, :2824)
    n = 512
    mods = R.coeff_modulus_create(n, [50, 40, 45, 60])
    assert mods == O.coeff_modulus_create(n, [50, 40, 45, 60])
    rc, oc = R.RefContext(R.CKKS, n, mods), O.Oracle(O.CKKS, n, mods)
    rng = np.random.default_rng(3)
    key = rc.relin_key()
    for i in range(len(mods)):
        a, _, c, d = rc.ntt_tables(i)
        root, rp, irp, invn = oc.ntt_tables(i)
        assert root == rc.ntt_root(i) and (a == rp).all() and (c == irp).all() and d == invn
    for L in (3, 2, 1):
        x, y = rand_ct(rng, mods, n, 2, L), rand_ct(rng, mods, n, 2, L)
        assert (rc.multiply_relin(L, x, y) == oc.multiply_relin(L, x, y, key)).all()
        if L > 1:
            assert (rc.rescale(L, x) == oc.rescale(L, x)).all()
        for step in (1, -5):
            e = rc.galois_elt_from_step(step)
            assert e == O.galois_elt_from_step(n, step)
            assert (rc.apply_galois(L, x, e) == oc.apply_galois(L, x, e, rc.galois_key(e))).all()


@needs_ref
def test_oracle_vs_live_reference_bfv_cfg1():
    # BASELINE.json configs[0]: BFV n=4096, 3x36-bit coeff_modulus, single multiply (bit-exact plumbing check)
    n = 4096
    mods = R.coeff_modulus_bfv_default(n)
    t = R.plain_modulus_batching(n, 20)
    rb, ob = R.RefContext(R.BFV, n, mods, t), O.Oracle(O.BFV, n, mods, t)
    rng = np.random.default_rng(4)
    L = 2
    assert rb.base_bsk(L) == ob.base_bsk(L)
    x, y = rand_ct(rng, mods, n, 2, L), rand_ct(rng, mods, n, 2, L)
    m = rb.multiply(L, x, y)
    assert (m == ob.multiply(L, x, y)).all()
    assert (rb.relinearize(L, m) == ob.relinearize(L, m, rb.relin_key())).all()
    e = rb.galois_elt_from_step(1)
    assert (rb.apply_galois(L, x, e) == ob.apply_galois(L, x, e, rb.galois_key(e))).all()


def test_oracle_linear_and_square_vs_live_reference():
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42])
    rc, oc = R.Replay(R.CKKS, n, mods), O.Oracle(O.CKKS, n, mods)
    rng = np.random.default_rng(21)
    L = 2
    a, b = rand_ct(rng, mods, n, 2, L), rand_ct(rng, mods, n, 2, L)
    for mode in (0, 1, 2):
        assert (rc.linear(mode, L, a, b) == oc.linear(mode, L, a, b)).all()
    assert (rc.square(L, a) == oc.multiply(L, a, a)).all()  # square computes the same residues as multiply(a, a)
    t = R.replay(R.plain_modulus_batching, n, 17)
    rb, ob = R.Replay(R.BFV, n, mods, t), O.Oracle(O.BFV, n, mods, t)
    assert (rb.square(L, a) == ob.multiply(L, a, a)).all()


@pytest.mark.parametrize("scheme", ["ckks", "bfv"])
def test_oracle_multiply_plain_vs_live_reference(scheme):
    # Evaluator::multiply_plain with ciphertext and plaintext both in NTT form (evaluator.cpp:2157-2195)
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42, 43])
    t = R.replay(R.plain_modulus_batching, n, 17) if scheme == "bfv" else 0
    sid = R.BFV if scheme == "bfv" else R.CKKS
    rc, oc = R.Replay(sid, n, mods, t), O.Oracle(sid, n, mods, t)
    rng = np.random.default_rng(23)
    for L in (3, 1):
        for size in (2, 3):
            a = rand_ct(rng, mods, n, size, L)
            plain = rand_ct(rng, mods, n, 1, L)[0]
            assert (rc.multiply_plain(L, a, plain) == oc.multiply_plain(L, a, plain)).all()


@needs_ref
@pytest.mark.parametrize("t_bits", [17, 38])
def test_oracle_vs_live_reference_bgv(t_bits):
    # SURVEY 8(f) rank 2: BGV branches -- bgv_multiply (evaluator.cpp:710-841), the BGV mod-down of switch_key_inplace
    # (:2762-2805) and mod_t_and_divide_q_last_ntt_inplace (rns.cpp:1193-1236); t above and below the coefficient primes
    n = 256
    mods = R.coeff_modulus_create(n, [40, 36, 42, 43])
    t = R.plain_modulus_batching(n, t_bits)
    rb, ob = R.RefContext(R.BGV, n, mods, t), O.Oracle(O.BGV, n, mods, t)
    rng = np.random.default_rng(29)
    key = rb.relin_key()
    for L in (3, 2, 1):
        a, b = rand_ct(rng, mods, n, 2, L), rand_ct(rng, mods, n, 2, L)
        m = rb.multiply(L, a, b)
        assert (m == ob.multiply(L, a, b)).all()
        assert (rb.relinearize(L, m) == ob.relinearize(L, m, key)).all()
        if L > 1:
            assert (rb.mod_switch(L, a) == ob.bgv_mod_switch(L, a)).all()
        e = rb.galois_elt_from_step(1)
        assert (rb.apply_galois(L, a, e) == ob.apply_galois(L, a, e, rb.galois_key(e))).all()


@pytest.mark.parametrize("scheme", ["ckks", "bfv", "bgv"])
def test_oracle_general_size_multiply_vs_live_reference(scheme):
    # the general-size branches of Evaluator::multiply (evaluator.cpp:524-560, :664-700, :796-833)
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42, 43])
    sid = {"ckks": R.CKKS, "bfv": R.BFV, "bgv": R.BGV}[scheme]
    t = 0 if scheme == "ckks" else R.replay(R.plain_modulus_batching, n, 17)
    rc, oc = R.Replay(sid, n, mods, t), O.Oracle(sid, n, mods, t)
    rng = np.random.default_rng(41)
    for L, sa, sb in ((3, 3, 2), (2, 2, 3), (1, 3, 3), (2, 4, 2)):
        a, b = rand_ct(rng, mods, n, sa, L), rand_ct(rng, mods, n, sb, L)
        assert (rc.multiply(L, a, b) == oc.multiply(L, a, b)).all()


@pytest.mark.parametrize("scheme,t_bits", [("bfv", 17), ("bfv", 38), ("bgv", 17), ("bgv", 38)])
def test_oracle_coeff_plain_ops_vs_live_reference(scheme, t_bits):
    # coefficient-form plaintexts: transform_to_ntt(Plaintext), multiply_plain (normal / NTT ciphertext), add_plain, sub_plain;
    # plain modulus below and above the smallest coefficient prime (fast and general plain lift, context.cpp:320-372)
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 36, 42, 43])
    t = R.replay(R.plain_modulus_batching, n, t_bits)
    sid = R.BFV if scheme == "bfv" else R.BGV
    rc, oc = R.Replay(sid, n, mods, t), O.Oracle(sid, n, mods, t)
    rng = np.random.default_rng(53)
    ntt = scheme == "bgv"
    for L in (3, 1):
        plain = rng.integers(0, t, n, dtype=np.uint64)
        plain[:4] = [0, t - 1, (t + 1) // 2, (t + 1) // 2 - 1]  # both sides of the upper-half threshold
        assert (rc.plain_to_ntt(L, plain) == oc.plain_to_ntt(L, plain)).all()
        for size in (2, 3):
            a = rand_ct(rng, mods, n, size, L)
            assert (rc.plain_op_coeff(0, L, a, plain, ntt) == oc.multiply_plain_coeff(L, a, plain, ntt)).all()
            if scheme == "bfv":  # a transformed BFV ciphertext takes the NTT branch (evaluator.cpp:1999-2004)
                assert (rc.plain_op_coeff(0, L, a, plain, True) == oc.multiply_plain_coeff(L, a, plain, True)).all()
            cf = 1 if scheme == "bfv" else 12345 % t
            assert (rc.plain_op_coeff(1, L, a, plain, ntt, cf) == oc.add_plain_coeff(L, a, plain, False, cf)).all()
            assert (rc.plain_op_coeff(2, L, a, plain, ntt, cf) == oc.add_plain_coeff(L, a, plain, True, cf)).all()


@pytest.mark.parametrize("scheme", ["bfv", "bgv"])
def test_oracle_batch_codec_vs_live_reference(scheme):
    # BatchEncoder::encode / decode (batchencoder.cpp:84-330)
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42])
    t = R.replay(R.plain_modulus_batching, n, 20)
    sid = R.BFV if scheme == "bfv" else R.BGV
    rc, oc = R.Replay(sid, n, mods, t), O.Oracle(sid, n, mods, t)
    rng = np.random.default_rng(61)
    v = rng.integers(0, t, n, dtype=np.uint64)
    p = rc.batch_codec(v, False)
    assert (p == oc.batch_codec(v, False)).all()
    assert (rc.batch_codec(p, True) == v).all() and (oc.batch_codec(p, True) == v).all()
    w = rng.integers(0, t, n, dtype=np.uint64)  # any coefficient vector decodes
    assert (rc.batch_codec(w, True) == oc.batch_codec(w, True)).all()


@pytest.mark.parametrize("scheme", ["ckks", "bfv", "bgv"])
def test_oracle_decrypt_vs_live_reference(scheme):
    # Decryptor::decrypt (decryptor.cpp): phase, then scale-and-round (BFV), exact base conversion (BGV) or nothing (CKKS);
    # uniform-random "ciphertexts" exercise every branch of the arithmetic
    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42, 43])
    sid = {"ckks": R.CKKS, "bfv": R.BFV, "bgv": R.BGV}[scheme]
    t = 0 if scheme == "ckks" else R.replay(R.plain_modulus_batching, n, 17)
    rc, oc = R.Replay(sid, n, mods, t), O.Oracle(sid, n, mods, t)
    sk = rc.secret_key()
    rng = np.random.default_rng(71)
    ntt = scheme != "bfv"
    for L, size in ((3, 2), (3, 3), (1, 2), (2, 4)):
        ct = rand_ct(rng, mods, n, size, L)
        cf = 1 if scheme != "bgv" else (12345 if size == 3 else 1)
        assert (rc.decrypt(L, ct, ntt, cf) == oc.decrypt(L, ct, sk, cf)).all()
    if scheme == "bfv":  # and a real encryption: decrypt(encrypt(m)) = m through both
        slots = rng.integers(0, t, n, dtype=np.uint64)
        ct = rc.bfv_encrypt(slots)
        p = oc.decrypt(3, ct, sk)
        assert (p == rc.decrypt(3, ct, False)).all()
        assert (oc.batch_codec(p, True) == slots).all()


@pytest.mark.skipif(not R.available(), reason="oracle/_ref/libsealref.so not present")
@pytest.mark.parametrize("scheme,n,bits", [("ckks", 4096, [40, 40, 40]), ("ckks", 8192, [60, 60, 60]), ("bfv", 4096, [36, 36, 37])])
def test_expand_seed_matches_reference_load(scheme, n, bits):
    """the oracle's restatement of Ciphertext::expand_seed (BLAKE2Xb stream + sample_poly_uniform with its rejection sampling,
    ciphertext.cpp:118-150, util/rlwe.cpp:104-132, randomgen.cpp:204-214) against the reference loading its own seeded stream"""
    import seal_b200 as S  # host-only use: the stream parser (no device needed)

    mods = R.coeff_modulus_create(n, bits)
    t = R.plain_modulus_batching(n, 20) if scheme == "bfv" else 0
    rc = R.RefContext(R.BFV if scheme == "bfv" else R.CKKS, n, mods, t)
    oc = O.Oracle(O.BFV if scheme == "bfv" else O.CKKS, n, mods, t)
    for _ in range(2):
        stream = rc.seeded_ct_stream()
        info = S.ciphertext_inspect(stream)
        assert info.seeded == 1 and info.size == 2 and info.seed_offset + 64 == len(stream)
        L = info.coeff_modulus_size
        full, _, _, _ = rc.ct_load(stream)  # the reference expands the seed itself
        c0 = np.frombuffer(stream, dtype=np.uint64, count=L * n, offset=info.data_offset).reshape(L, n)
        seed = np.frombuffer(stream, dtype=np.uint64, count=8, offset=info.seed_offset)
        assert (full[0] == c0).all()
        assert (oc.expand_seed(L, seed) == full[1]).all()


@pytest.mark.skipif(not R.available(), reason="oracle/_ref/libsealref.so not present")
@pytest.mark.parametrize("scheme,n,bits", [("ckks", 4096, [40, 40, 40]), ("bfv", 4096, [36, 36, 37]), ("bgv", 4096, [40, 40, 40]),
                                          ("ckks", 2048, [54])])
def test_encrypt_zero_symmetric_matches_reference(scheme, n, bits):
    """the oracle's restatement of encrypt_zero_symmetric (util/rlwe.cpp:264-408: public seed + uniform c_1 from one PRNG, centred
    binomial noise from the bootstrap PRNG, c_0 = -(c_1 s + e)) against the reference's Encryptor with the same bootstrap seed,
    both the plain and the seed-compressed variant (they differ for BFV)"""
    sid = {"ckks": R.CKKS, "bfv": R.BFV, "bgv": R.BGV}[scheme]
    mods = R.coeff_modulus_create(n, bits)
    t = R.plain_modulus_batching(n, 20) if scheme != "ckks" else 0
    seed0 = 0x5EA1
    rc = R.RefContext(sid, n, mods, t, seed=seed0)
    oc = O.Oracle({"ckks": O.CKKS, "bfv": O.BFV, "bgv": O.BGV}[scheme], n, mods, t)
    sk = rc.secret_key()
    seed = np.zeros(8, dtype=np.uint64)
    seed[0] = seed0
    assert (oc.encrypt_zero_symmetric(sk, seed, False) == rc.encrypt_zero_symmetric()).all()
    seeded, _, _, _ = rc.ct_load(rc.seeded_ct_stream())
    assert (oc.encrypt_zero_symmetric(sk, seed, True) == seeded).all()
    if len(mods) > 2:  # a lower level: sampled at that level directly (no modulus switching for symmetric encryption)
        assert (oc.encrypt_zero_symmetric(sk, seed, False, L=1) == rc.encrypt_zero_symmetric(L=1)).all()


@pytest.mark.parametrize("n,bits", [(4096, [40, 40, 40]), (1024, [27]), (8192, [60, 60, 60, 60]), (2048, [54])])
def test_ckks_encoder_matches_reference(n, bits):
    """the oracle's CKKSEncoder restatement (ckks.h:455-807; double-precision FFT in the reference's operation order) is BIT-exact
    against the reference: full and partial vectors, scales that reach the 64-bit, 128-bit and multi-precision decomposition
    branches, lower levels, the error cases, and decode of encoded and of arbitrary plaintexts"""
    mods = R.replay(R.coeff_modulus_create, n, bits)
    rc = R.Replay(R.CKKS, n, mods)
    oc = O.Oracle(O.CKKS, n, mods)
    k = len(mods)
    Lmax = k - 1 if k > 1 else 1
    rng = np.random.default_rng(7)
    slots = n // 2
    total = sum(bits[:Lmax])
    cases = [(Lmax, slots, 2.0 ** 20, 1.0), (Lmax, slots // 3, 2.0 ** 30, 100.0), (1, slots, 2.0 ** 10, 1e-3), (Lmax, 0, 2.0 ** 20, 1.0),
             (Lmax, 1, 3.7e5, 1.0)]
    if total > 70:
        cases.append((Lmax, slots, 2.0 ** 62, 50.0))     # coefficients beyond 64 bits
    if total > 140:
        cases.append((Lmax, slots, 2.0 ** 120, 1000.0))  # beyond 128 bits: the multi-precision branch
    for L, count, scale, mag in cases:
        v = (rng.standard_normal(count) + 1j * rng.standard_normal(count)) * mag
        want = rc.ckks_encode(L, v, scale)
        got = oc.ckks_encode(L, v, scale)
        assert (want is None) == (got is None), (L, count, scale)
        if want is None:
            continue
        assert (got == want).all(), (L, count, scale)
        dw, dg = rc.ckks_decode(L, want, scale), oc.ckks_decode(L, got, scale)  # got has want's words (asserted above)
        assert dw is not None and dg is not None
        assert (dw.view(np.uint64) == dg.view(np.uint64)).all(), ("decode", L, count, scale)
        if count and scale >= 2.0 ** 20:
            assert np.abs(dg[:count] - v).max() < mag * 1e-3 + 1e-3
    # error cases: values too large for the modulus, non-finite input, scale out of bounds
    assert rc.ckks_encode(1, np.full(slots, 1e30 + 0j), 2.0 ** 20) is None and oc.ckks_encode(1, np.full(slots, 1e30 + 0j), 2.0 ** 20) is None
    assert oc.ckks_encode(1, np.array([np.inf + 0j]), 2.0 ** 20) is None and rc.ckks_encode(1, np.array([np.inf + 0j]), 2.0 ** 20) is None
    assert oc.ckks_encode(1, np.ones(4) + 0j, 2.0 ** 200) is None and rc.ckks_encode(1, np.ones(4) + 0j, 2.0 ** 200) is None
    # decode of an arbitrary plaintext (uniform residues: large "negative" and positive coefficients)
    for L in sorted({1, Lmax}):
        p = np.stack([rng.integers(0, mods[j], n, dtype=np.uint64) for j in range(L)])
        for scale in (2.0 ** 12, 2.0 ** 30):
            dw, dg = rc.ckks_decode(L, p, scale), oc.ckks_decode(L, p, scale)
            assert (dw is None) == (dg is None), ("decode random: scale bound", L, scale)
            assert dw is None or (dw.view(np.uint64) == dg.view(np.uint64)).all(), ("decode random", L, scale)


@pytest.mark.skipif(not R.available(), reason="oracle/_ref/libsealref.so not present")
@pytest.mark.parametrize("scheme,n,bits", [("ckks", 4096, [40, 40, 40, 40]), ("bfv", 4096, [36, 36, 37]), ("bgv", 4096, [40, 40, 40]),
                                          ("ckks", 2048, [54])])
def test_encrypt_zero_asymmetric_matches_reference(scheme, n, bits):
    """the oracle's restatement of public-key encryption of zero (ternary u through libstdc++'s uniform_int_distribution, two noise
    polynomials, c_j = pk_j u + e_j one level up, divide-and-round down) against Encryptor(public key)::encrypt_zero with the same
    PRNG seed: first data level, a lower level, the key level"""
    sid = {"ckks": R.CKKS, "bfv": R.BFV, "bgv": R.BGV}[scheme]
    mods = R.coeff_modulus_create(n, bits)
    t = R.plain_modulus_batching(n, 20) if scheme != "ckks" else 0
    seed0 = 0x5EA1
    rc = R.RefContext(sid, n, mods, t, seed=seed0)
    oc = O.Oracle({"ckks": O.CKKS, "bfv": O.BFV, "bgv": O.BGV}[scheme], n, mods, t)
    pk = rc.public_key()
    seed = np.zeros(8, dtype=np.uint64)
    seed[0] = seed0
    k = len(mods)
    levels = sorted({k - 1 if k > 1 else 1, 1, k})
    for L in levels:
        assert (oc.encrypt_zero_asymmetric(pk, seed, L=L) == rc.encrypt_zero_asymmetric(L=L)).all(), L
