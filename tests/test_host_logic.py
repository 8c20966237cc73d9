"""CPU-side tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/seal_b200.h declares (no
compute calls without a GPU), host helpers agree with the oracle, the shared-memory swizzle used by the local NTT pass
is bank-conflict free, and the multi-GPU sharding logic works under a world_size-2 gloo group."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def test_library_exports_every_declared_symbol():
    import seal_b200

    hdr = open(os.path.join(ROOT, "include", "seal_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", hdr)))
    assert declared, "no declarations parsed"
    assert sorted(seal_b200.SYMBOLS) == declared
    lib = seal_b200.lib()  # must exist and load on a box without a GPU
    for s in declared:
        assert getattr(lib, s) is not None


def test_no_gpu_means_loud_failure_not_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import seal_b200

    with pytest.raises(RuntimeError) as e:
        seal_b200.Context(seal_b200.CKKS, 1024, O.coeff_modulus_create(1024, [40, 40]))
    assert "no CUDA device" in str(e.value) or "CUDA" in str(e.value)


def test_coeff_modulus_create_matches_oracle():
    import seal_b200

    for n, bits in [(4096, [36, 36, 37]), (8192, [54] * 4), (65536, [55] * 8), (1024, [20, 30, 20, 40])]:
        assert seal_b200.coeff_modulus_create(n, bits) == O.coeff_modulus_create(n, bits)
    with pytest.raises(ValueError):
        seal_b200.coeff_modulus_create(1000, [40])
    with pytest.raises(ValueError):
        seal_b200.coeff_modulus_create(1024, [61])


def test_swizzle_conflict_free():
    # sb_ntt.cuh::swz -- every access pattern of the warp-local passes must hit 16 distinct 8-byte banks per half-warp
    def swz(e):
        b4, b5, b6 = (e >> 4) & 1, (e >> 5) & 1, (e >> 6) & 1
        return e ^ (b4 | (b5 << 1) | (b6 << 2) | ((b5 ^ b6) << 3))

    pats = [lambda l, j: l + 32 * j, lambda l, j: 32 * (l >> 2) + (l & 3) + 4 * j, lambda l, j: 8 * l + j,
            lambda l, j: 64 * (l >> 3) + (l & 7) + 8 * j]
    for f in pats:
        assert sorted(swz(f(l, j)) for l in range(32) for j in range(8)) == list(range(256))
        for j in range(8):
            for half in (0, 16):
                assert len({swz(f(l, j)) % 16 for l in range(half, half + 16)}) == 16


def test_shard_range_partitions_batch():
    from seal_b200.shard import shard_range

    for batch in (1, 7, 8, 8192, 1000):
        for world in (1, 2, 3, 8):
            cover = []
            for r in range(world):
                lo, hi = shard_range(batch, r, world)
                cover += list(range(lo, hi))
            assert cover == list(range(batch))


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from seal_b200.shard import shard_range, digest, gather_digests
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
batch = 7
g = torch.Generator().manual_seed(1)
full = torch.randint(-2**62, 2**62, (batch, 2, 3, 16), generator=g, dtype=torch.int64)   # the global "output slab"
lo, hi = shard_range(batch, rank, world)
d = gather_digests(digest(full[lo:hi]), rank, world)
if rank == 0:
    assert torch.equal(d, digest(full)), "gathered digests differ from the unsharded run"
    print("GATHER_OK")
dist.destroy_process_group()
"""


def test_multi_rank_gather_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29611", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), os.path.abspath(ROOT)], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GATHER_OK" in outs[0][0]


# ---- the product's host-side precomputation (sb_host.cpp) against the oracle, on the CPU ---------------------------
def _probe():
    import ctypes as C

    d = os.path.join(ROOT, "tests", "cpp")
    subprocess.check_call(["make", "-C", d, "probe"], stdout=subprocess.DEVNULL)
    L = C.CDLL(os.path.join(d, "_bin", "libhostprobe.so"))
    u64p = C.POINTER(C.c_uint64)
    L.probe_tables.argtypes = [C.c_size_t, C.c_uint64] + [u64p] * 8
    L.probe_bsk.restype = C.c_size_t
    L.probe_bsk.argtypes = [C.c_size_t, u64p, C.c_size_t, C.c_uint64, u64p]
    L.probe_galois_table.argtypes = [C.c_size_t, C.c_uint32, C.POINTER(C.c_uint32)]
    L.probe_elt_from_step.restype = C.c_uint32
    L.probe_elt_from_step.argtypes = [C.c_size_t, C.c_int]
    L.probe_is_prime.argtypes = [C.c_uint64]
    L.probe_parms_id.argtypes = [C.c_int, C.c_size_t, u64p, C.c_size_t, C.c_uint64, u64p]
    L.probe_blake2b_256.argtypes = [C.c_char_p, C.c_size_t, u64p]
    L.probe_batch_index_map.argtypes = [C.c_size_t, C.POINTER(C.c_uint32)]
    L.probe_kswitch_offsets.restype = C.c_long
    L.probe_kswitch_offsets.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.c_size_t, C.POINTER(C.c_size_t),
                                        C.POINTER(C.c_size_t)]
    return L


def _pp(a):
    import ctypes as C

    return a.ctypes.data_as(C.POINTER(C.c_uint64))


@pytest.mark.parametrize("n,bits", [(2, None), (8, [20]), (1024, [40, 50]), (4096, [36, 60]), (32768, [55])])
def test_host_tables_match_oracle(n, bits):
    import ctypes as C

    P = _probe()
    mods = [0xFFFFFFFFFFC0001] if bits is None else O.coeff_modulus_create(n, bits)
    oc = O.Oracle(O.CKKS, n, mods)
    for i, q in enumerate(mods):
        root, inv_n = C.c_uint64(0), C.c_uint64(0)
        rp, rpq, irp, fw, iw = (np.zeros(n, dtype=np.uint64) for _ in range(5))
        ratio = np.zeros(2, dtype=np.uint64)
        assert P.probe_tables(n, q, C.byref(root), _pp(rp), _pp(rpq), _pp(irp), C.byref(inv_n), _pp(fw), _pp(iw), _pp(ratio)) == 0
        oroot, orp, oirp, oinv = oc.ntt_tables(i)
        assert root.value == oroot and (rp == orp).all() and (irp == oirp).all() and inv_n.value == oinv
        # Shoup quotients and the Barrett ratio are exact floors
        for j in (0, 1, n // 2, n - 1):
            assert int(rpq[j]) == (int(rp[j]) << 64) // q
        assert (int(ratio[1]) << 64) + int(ratio[0]) == (1 << 128) // q
        # device order: fwd[m+i] = root_powers[m+i]; inv[m+i] = inv_root_powers[n-2m+1+i]
        assert (fw == rp).all()
        m = 1
        while m < n:
            assert (iw[m:2 * m] == irp[n - 2 * m + 1:n - m + 1]).all()
            m *= 2
    if n == 2:  # native/tests/seal/util/ntt.cpp:53-63
        assert int(rp[1]) == 288794978602139552


def test_host_galois_and_behz_match_oracle():
    import ctypes as C

    P = _probe()
    # native/tests/seal/util/galois.cpp:104-120: n=8, g=3 -> NTT-form permutation {4,5,7,6,1,0,2,3}
    t = np.zeros(8, dtype=np.uint32)
    P.probe_galois_table(8, 3, t.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert list(t) == [4, 5, 7, 6, 1, 0, 2, 3]
    x = np.arange(8, dtype=np.uint64)
    assert list(x[t]) == list(O.galois_ntt_row(8, 3, x))
    for n in (8, 4096, 65536):
        for step in (0, 1, -1, 3, -(n // 2 - 1), n // 2 - 1):
            assert P.probe_elt_from_step(n, step) == O.galois_elt_from_step(n, step)
        assert P.probe_elt_from_step(n, n // 2) == 0  # "step count too large" (galois.cpp:72-75)
    n = 4096
    for q, tt in (([0xFFFFEE001, 0xFFFFC4001], 1032193), (O.coeff_modulus_create(n, [60, 60, 60])[:2], 1 << 30)):
        out = np.zeros(8, dtype=np.uint64)
        cnt = P.probe_bsk(n, _pp(np.array(q, dtype=np.uint64)), len(q), tt, _pp(out))
        assert [int(v) for v in out[:cnt]] == O.behz_base(n, q, tt)
    assert P.probe_is_prime(0xFFFFEE001) == 1 and P.probe_is_prime(0xFFFFEE003) == O.lib().orc_is_prime(0xFFFFEE003)


# ---- wire format (SURVEY 8f rank 3): parms_id hashing and stream parsing are pure host code ---------------------------
def test_blake2b_matches_hashlib():
    import hashlib

    P = _probe()
    rng = np.random.default_rng(5)
    for ln in (0, 1, 24, 127, 128, 129, 256, 1000):
        msg = rng.integers(0, 256, ln, dtype=np.uint8).tobytes()
        out = np.zeros(4, dtype=np.uint64)
        P.probe_blake2b_256(msg, ln, _pp(out))
        assert out.tobytes() == hashlib.blake2b(msg, digest_size=32).digest()


@pytest.mark.parametrize("scheme", ["bfv", "ckks", "bgv"])
def test_parms_id_matches_reference(scheme):
    import refseal as R

    P = _probe()
    n = 1024
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42, 43])
    sid = {"bfv": R.BFV, "ckks": R.CKKS, "bgv": R.BGV}[scheme]
    t = 0 if scheme == "ckks" else R.replay(R.plain_modulus_batching, n, 17)
    rc = R.Replay(sid, n, mods, t)
    q = np.array(mods, dtype=np.uint64)
    for L in (4, 3, 2, 1):  # 4 = the key level
        out = np.zeros(4, dtype=np.uint64)
        P.probe_parms_id(sid, n, _pp(q), L, t, _pp(out))
        assert tuple(int(x) for x in out) == rc.parms_id(L)


def test_ciphertext_inspect_vs_reference_stream():
    import refseal as R
    import seal_b200 as S
    from common import rand_ct

    n = 256
    mods = R.replay(R.coeff_modulus_create, n, [40, 41, 42])
    rc = R.Replay(R.CKKS, n, mods)
    rng = np.random.default_rng(6)
    for L, size in ((2, 2), (1, 3)):
        data = rand_ct(rng, mods, n, size, L)
        stream = rc.ct_save(L, data, True, scale=2.0 ** 30, correction_factor=1)
        info = S.ciphertext_inspect(stream)
        assert tuple(info.parms_id) == rc.parms_id(L)
        assert (info.size, info.poly_modulus_degree, info.coeff_modulus_size) == (size, n, L)
        assert info.is_ntt_form == 1 and info.seeded == 0 and info.scale == 2.0 ** 30 and info.correction_factor == 1
        assert info.stream_bytes == len(stream) and info.data_words == data.size
        words = np.frombuffer(stream, dtype=np.uint64, count=data.size, offset=info.data_offset)
        assert (words == data.reshape(-1)).all()
    # seed-compressed ciphertexts: the PRNG type and where the seed sits
    sinfo = S.ciphertext_inspect(rc.seeded_ct_stream())
    assert sinfo.seeded == 1 and sinfo.seed_offset + 64 == sinfo.stream_bytes and sinfo.compr_mode == 0
    # zlib-compressed objects (compr_mode_type::zlib) are inflated on the host and parse to the same metadata and words
    z = rc.ct_save(L, data, True, scale=2.0 ** 30, correction_factor=1, compr=1)
    assert z[5] == 1 and len(z) != len(stream)
    zinfo = S.ciphertext_inspect(z)
    assert zinfo.compr_mode == 1 and zinfo.stream_bytes == len(z) and zinfo.data_words == data.size and tuple(zinfo.parms_id) == rc.parms_id(L)
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(z[:40] + bytes([z[40] ^ 0xFF]) + z[41:])   # corrupted deflate data
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(z[:len(z) // 2] + b"\x00" * (len(z) - len(z) // 2))  # truncated deflate data
    # malformed streams: Serialization::Load's error ladder
    with pytest.raises(ValueError):
        S.ciphertext_inspect(stream[:8])                       # insufficient size
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(b"\x00\x00" + stream[2:])         # bad magic
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(stream[:3] + b"\x05" + stream[4:])  # newer major version
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(stream[:5] + b"\x02" + stream[6:])  # compressed
    with pytest.raises(RuntimeError):
        S.ciphertext_inspect(stream[:-8])                      # truncated


@pytest.mark.skipif(not __import__("refseal").available(), reason="oracle/_ref not built")
def test_kswitch_keys_stream_parsing_vs_reference():
    # KSwitchKeys::save layout (kswitchkeys.cpp:42-86): the product locates data()[index][j] inside the stream
    import ctypes as C

    import refseal as R

    P = _probe()
    n = 256
    mods = R.coeff_modulus_create(n, [40, 41, 42, 43])
    k = len(mods)
    rc = R.RefContext(R.CKKS, n, mods)

    def entry(stream, index):
        offs = (C.c_size_t * 16)()
        L, nn = C.c_size_t(0), C.c_size_t(0)
        d = P.probe_kswitch_offsets(stream, len(stream), index, offs, 16, C.byref(L), C.byref(nn))
        if d < 0:
            return d
        assert (L.value, nn.value) == (k, n)
        return np.stack([np.frombuffer(stream, dtype=np.uint64, count=2 * k * n, offset=offs[j]).reshape(2, k, n) for j in range(d)])

    rs = rc.kswitch_keys_stream(0)
    assert (entry(rs, 0) == rc.relin_key()).all()
    assert entry(rs, 1) == -3  # out of range: RelinKeys made for size-3 ciphertexts hold one entry
    e = rc.galois_elt_from_step(1)
    gs = rc.kswitch_keys_stream(e)
    assert (entry(gs, (e - 1) // 2) == rc.galois_key(e)).all()
    assert entry(gs, 0) == -1  # an empty slot: "key not present"
    assert entry(gs[:200], (e - 1) // 2) == -2  # truncated


def test_batch_index_map_matches_oracle():
    # BatchEncoder::populate_matrix_reps_index_map (batchencoder.cpp:54-76): encode = scatter by the map + INTT modulo t
    import ctypes as C

    P = _probe()
    for n, t in ((8, 17), (256, 12289), (4096, 1032193)):
        m = np.zeros(n, dtype=np.uint32)
        P.probe_batch_index_map(n, m.ctypes.data_as(C.POINTER(C.c_uint32)))
        assert sorted(m) == list(range(n))
        oc = O.Oracle(O.BFV, n, O.coeff_modulus_create(n, [30, 31]), t)
        rng = np.random.default_rng(n)
        v = rng.integers(0, t, n, dtype=np.uint64)
        scattered = np.zeros(n, dtype=np.uint64)
        scattered[m] = v
        # decode(plain)[i] = NTT_t(plain)[map[i]]: the scattered vector is the transform of encode(v)
        assert (oc.batch_codec(oc.batch_codec(v, False), True) == v).all()
        tt = O.Oracle(O.CKKS, n, [t])  # a context whose only prime is t gives the plain transform
        assert (tt.ntt_row(0, oc.batch_codec(v, False)) == scattered).all()


@pytest.mark.parametrize("args", [["4096", "36", "36", "37"], ["8192", "55", "55", "55", "56"], ["16384", "60", "60", "60"],
                                  ["32768"] + ["55"] * 16])
def test_ksint_host_tables_transforms_and_crt(args):
    """integer key-switching path (seal_b200/csrc/sb_ksint.cu): the tables sbh::build_ksint produces, driven on the CPU with
    the kernels' own index scheme, give transforms that invert each other and satisfy the convolution theorem, and CRT
    constants that reconstruct signed integers inside the bound L n q^2 exactly (tests/cpp/ksint_host_check.cpp)"""
    cpp = os.path.join(ROOT, "tests", "cpp")
    subprocess.check_call(["make", "-C", cpp, "ksint"], stdout=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(cpp, "_bin", "ksint_host_check")] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_ksint_swizzle_conflict_free():
    """shared-memory layout of the 4096-word blocks of the 32-bit local passes (swz32 in sb_ksint.cu): every access pattern of
    the three radix-16 passes touches 32 distinct banks per warp-wide 4-byte access and 8 distinct 16-byte bank groups per
    quarter-warp for the 16-byte accesses of the last pass"""
    def swz(i):
        return i ^ (((i >> 8) & 1) << 4) ^ (((i >> 5) & 3) << 2)

    assert sorted(swz(i) for i in range(4096)) == list(range(4096))
    for warp in range(8):
        tids = [warp * 32 + l for l in range(32)]
        for e in range(16):
            assert len({swz(t + 256 * e) % 32 for t in tids}) == 32                              # pass 1
            assert len({swz(((t >> 4) << 8) + (t & 15) + 16 * e) % 32 for t in tids}) == 32      # pass 2
        for h in range(4):                                                                        # pass 3: 16-byte accesses
            for q in range(4):
                grp = tids[8 * q: 8 * q + 8]
                phys = [((16 * t) ^ (((t >> 4) & 1) << 4)) + 4 * (h ^ ((t >> 1) & 3)) for t in grp]
                assert all(p == swz(16 * t + 4 * h) for p, t in zip(phys, grp))
                assert len({(p // 4) % 8 for p in phys}) == 8


@pytest.mark.parametrize("scheme", ["ckks", "bfv"])
def test_integer_key_switching_identity_vs_oracle(scheme):
    """the identity the integer key-switching path rests on (seal_b200/csrc/sb_ksint.cuh), checked with Python integers against the
    oracle's switch_key_inplace restatement at n = 16: the digit sum sum_J NTT_I(d_J) (.) K_JI is the NTT_I image of the INTEGER
    polynomial sum_J d_J * INTT_I(K_JI) reduced mod q_I; reconstructing that integer from its residues modulo 29-bit primes (with the
    offset P/2 and alpha = floor(sum y_t / p_t)) and doing the mod-down in coefficient form gives the reference's words"""
    n, bits = 16, [40, 40, 40, 41]
    mods = O.coeff_modulus_create(n, bits)
    k, L = len(mods), len(mods) - 1
    sid = O.CKKS if scheme == "ckks" else O.BFV
    oc = O.Oracle(sid, n, mods, 0 if scheme == "ckks" else 65537)
    rng = np.random.default_rng(5)
    c3 = np.stack([np.stack([rng.integers(0, mods[i], n, dtype=np.uint64) for i in range(L)]) for _ in range(3)])
    key = np.stack([np.stack([np.stack([rng.integers(0, mods[i], n, dtype=np.uint64) for i in range(k)]) for _ in range(2)])
                    for _ in range(L)])
    want = oc.relinearize(L, c3, key)

    def negconv(a, b):
        r = [0] * n
        for i in range(n):
            for j in range(n):
                if i + j < n:
                    r[i + j] += a[i] * b[j]
                else:
                    r[i + j - n] -= a[i] * b[j]
        return r

    # digits: coefficient form of the target (CKKS: INTT per prime; BFV: already coefficients)
    D = [[int(v) for v in (oc.intt_row(J, c3[2][J]) if scheme == "ckks" else c3[2][J])] for J in range(L)]
    aux, cand = [], ((1 << 29) // (2 * n)) * (2 * n) + 1
    while len(aux) < 5:  # the largest 29-bit primes = 1 mod 2n, as sbh::build_ksint picks them
        cand -= 2 * n
        if all(cand % d for d in range(3, 23171, 2)):
            aux.append(cand)
    P = 1
    for p in aux:
        P *= p
    H = (P - 1) // 2
    assert P > 4 * L * n * max(mods) ** 2
    qsp, half = int(mods[k - 1]), int(mods[k - 1]) >> 1
    out = np.zeros((2, L, n), dtype=np.uint64)
    for comp in range(2):
        A = {}
        for I in list(range(L)) + [k - 1]:
            q = int(mods[I])
            acc = [0] * n
            for J in range(L):
                kI = [int(v) for v in oc.intt_row(I, key[J][comp][I])]
                acc = [x + y for x, y in zip(acc, negconv(D[J], kI))]
            res = []
            for x in range(n):
                assert abs(acc[x]) < P // 4
                y = [((acc[x] + H) % p) * pow(P // p, -1, p) % p for p in aux]
                alpha = sum(yt * ((1 << 60) // p) for yt, p in zip(y, aux)) >> 60  # the kernels' estimate of floor(sum y_t / p_t)
                assert alpha == sum(yt * (P // p) for yt, p in zip(y, aux)) // P
                v = (sum(yt * ((P // p) % q) for yt, p in zip(y, aux)) - alpha * (P % q) - H % q) % q
                assert v == acc[x] % q
                res.append(v)
            A[I] = res
        for i in range(L):
            q = int(mods[i])
            inv = pow(qsp, -1, q)
            r = [((A[i][x] - ((A[k - 1][x] + half) % qsp % q - half % q)) * inv) % q for x in range(n)]
            if scheme == "ckks":
                r = [int(v) for v in oc.ntt_row(i, np.array(r, dtype=np.uint64))]
            out[comp][i] = [(r[x] + int(c3[comp][i][x])) % q for x in range(n)]
    assert (out == want).all()


def test_one_word_barrett_bound():
    """barrett_wide (seal_b200/csrc/sb_device.cuh): for z < 2^(b+62), b = bit length of q, the quotient estimate
    floor(floor(z / 2^(b-2)) * floor(2^(b+62) / q) / 2^64) is at most 2 below floor(z / q), so z - t q lies in [0, 3q) and its low
    64 bits are the whole value: the two conditional subtractions of the kernel canonicalise it.  Python-integer re-enactment."""
    rng = np.random.default_rng(62)
    for _ in range(4000):
        b = int(rng.integers(2, 62))
        q = int(rng.integers(1 << (b - 1), 1 << b)) | 1
        if q.bit_length() != b:
            continue
        mu, sh = (1 << (b + 62)) // q, b - 2
        assert mu < 1 << 63
        for z in (int(rng.integers(0, 1 << 62)) * (1 << b) // (1 << int(rng.integers(0, 62))), (1 << (b + 62)) - 1, q * q - 1 if b <= 61 else 0,
                  2 * (q - 1) ** 2):
            if z >= 1 << (b + 62):
                continue
            zh = z >> sh
            assert zh < 1 << 64
            t = (zh * mu) >> 64
            r = z - t * q
            assert 0 <= r < 3 * q and r < 1 << 64, (b, q, z)
            assert (z & ((1 << 64) - 1)) - ((t * q) & ((1 << 64) - 1)) in (r, r - (1 << 64))  # what the 64-bit subtraction yields
