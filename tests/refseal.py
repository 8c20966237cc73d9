"""ctypes driver for oracle/_ref/libsealref.so -- the UNMODIFIED reference (microsoft/SEAL 4.4.3) behind the flat
C wrapper oracle/ref_capi.{h,cpp}.  TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs; the product never loads it.
"""
import atexit
import base64
import ctypes as C
import hashlib
import json
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "..", "oracle", "_ref", "libsealref.so")
_RECORDED_PATH = os.path.join(_HERE, "golden", "reference_results.json")

BFV, CKKS, BGV = 1, 2, 3
_u64p = C.POINTER(C.c_uint64)


def available():
    return os.path.exists(_LIB_PATH)


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_LIB_PATH)
        L.sealref_create.restype = C.c_void_p
        L.sealref_create.argtypes = [C.c_int, C.c_size_t, _u64p, C.c_size_t, C.c_uint64, C.c_uint64]
        L.sealref_destroy.argtypes = [C.c_void_p]
        L.sealref_last_error.restype = C.c_char_p
        L.sealref_coeff_modulus_create.argtypes = [C.c_size_t, C.POINTER(C.c_int), C.c_size_t, _u64p]
        L.sealref_coeff_modulus_bfv_default.argtypes = [C.c_size_t, _u64p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.sealref_plain_modulus_batching.restype = C.c_uint64
        L.sealref_plain_modulus_batching.argtypes = [C.c_size_t, C.c_int]
        L.sealref_ntt_root.argtypes = [C.c_void_p, C.c_size_t, _u64p]
        L.sealref_ntt_tables.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p, _u64p, _u64p]
        L.sealref_base_bsk.restype = C.c_size_t
        L.sealref_base_bsk.argtypes = [C.c_void_p, C.c_size_t, _u64p, C.c_size_t]
        L.sealref_relin_key.argtypes = [C.c_void_p, _u64p]
        L.sealref_galois_key.argtypes = [C.c_void_p, C.c_uint32, _u64p]
        L.sealref_galois_elt_from_step.restype = C.c_uint32
        L.sealref_galois_elt_from_step.argtypes = [C.c_void_p, C.c_int]
        L.sealref_ntt_forward.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p]
        L.sealref_ntt_inverse.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p]
        L.sealref_multiply.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p, _u64p]
        L.sealref_square.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p]
        L.sealref_multiply_sized.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, _u64p, _u64p, _u64p]
        L.sealref_linear.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, _u64p, _u64p, _u64p]
        L.sealref_multiply_plain_ntt.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p, _u64p, _u64p]
        L.sealref_relinearize.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p]
        L.sealref_multiply_relin.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p, _u64p]
        L.sealref_rescale.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p]
        L.sealref_mod_switch.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p]
        L.sealref_apply_galois.argtypes = [C.c_void_p, C.c_size_t, _u64p, C.c_uint32, _u64p]
        L.sealref_rotate.argtypes = [C.c_void_p, C.c_size_t, _u64p, C.c_int, _u64p]
        L.sealref_bfv_encrypt.argtypes = [C.c_void_p, _u64p, _u64p]
        L.sealref_bfv_decrypt.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p, _u64p, C.POINTER(C.c_int)]
        L.sealref_time_op.restype = C.c_double
        L.sealref_time_op.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int]
        L.sealref_batch_codec.argtypes = [C.c_void_p, C.c_int, _u64p, _u64p]
        L.sealref_secret_key.argtypes = [C.c_void_p, _u64p]
        L.sealref_decrypt.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_uint64, _u64p, _u64p]
        L.sealref_plain_to_ntt.argtypes = [C.c_void_p, C.c_size_t, _u64p, _u64p]
        L.sealref_plain_op_coeff.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_uint64, _u64p, _u64p, _u64p]
        L.sealref_parms_id.argtypes = [C.c_void_p, C.c_size_t, _u64p]
        L.sealref_ct_save.restype = C.c_long
        L.sealref_ct_save.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p, C.c_int, C.c_double, C.c_uint64, C.c_char_p, C.c_size_t]
        L.sealref_ct_load.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, _u64p, C.c_size_t, _u64p, _u64p, C.POINTER(C.c_int),
                                      C.POINTER(C.c_double), _u64p]
        L.sealref_kswitch_keys_stream.restype = C.c_long
        L.sealref_kswitch_keys_stream.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_size_t]
        L.sealref_seeded_ct_stream.restype = C.c_long
        L.sealref_seeded_ct_stream.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
        L.sealref_ckks_encode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_double, _u64p]
        L.sealref_ckks_decode.argtypes = [C.c_void_p, C.c_size_t, _u64p, C.c_double, C.c_void_p]
        L.sealref_public_key.argtypes = [C.c_void_p, _u64p]
        L.sealref_encrypt_zero_asymmetric.argtypes = [C.c_void_p, C.c_size_t, _u64p]
        L.sealref_encrypt_zero_symmetric.argtypes = [C.c_void_p, C.c_size_t, _u64p]
        L.sealref_ct_save_mode.restype = C.c_long
        L.sealref_ct_save_mode.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, _u64p, C.c_int, C.c_double, C.c_uint64, C.c_int, C.c_char_p, C.c_size_t]
        L.sealref_kswitch_keys_stream_mode.restype = C.c_long
        L.sealref_kswitch_keys_stream_mode.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_size_t]
        L.sealref_seeded_ct_stream_mode.restype = C.c_long
        L.sealref_seeded_ct_stream_mode.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t]
        _lib = L
    return _lib


def _p(a):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_u64p)


# ------------------------------------------------------------------------------------------- recorded results ----
# Tests that only compare with the reference's results run everywhere: through Replay, a call is answered by the live library
# when oracle/_ref is built, and otherwise from tests/golden/reference_results.json, which holds, per call (keyed by the context,
# the method and a digest of every argument), the SHA-256 digest of the result, and the result itself for the methods whose
# results the tests feed to other code (_DATA_METHODS).  A digest-only result (Recorded) compares equal to exactly the words the
# reference returned.  With SEAL_B200_RECORD_REFERENCE=1 and the live library, the calls a test run makes are added to the file;
# a live result that contradicts the file fails.
_DATA_METHODS = {"secret_key", "bfv_encrypt", "batch_codec", "ct_save", "seeded_ct_stream"}
_recorded = None
_record = os.environ.get("SEAL_B200_RECORD_REFERENCE") == "1"


def _bytes_digest(b):
    return hashlib.sha256(b).hexdigest()[:40]


class Recorded:
    """A reference result known by the digest of its bytes only; `x == recorded` is true iff x has exactly those bytes"""

    __array_ufunc__ = None  # ndarray == Recorded defers to Recorded.__eq__
    __hash__ = None

    def __init__(self, digest):
        self.digest = digest

    def view(self, *_):  # the digest covers the raw bytes, whatever dtype they are viewed as
        return self

    def __eq__(self, other):
        return _Match(_digest_of(other) == self.digest)

    def __ne__(self, other):
        return _Match(_digest_of(other) != self.digest)


class _Match:
    def __init__(self, ok):
        self.ok = ok

    def all(self):
        return self.ok


def _digest_of(x):
    if isinstance(x, Recorded):
        return x.digest
    if isinstance(x, bytes):
        return _bytes_digest(x)
    return _bytes_digest(np.ascontiguousarray(x).tobytes())


def _encode(r, full):
    if r is None:
        return {"none": 1}
    if isinstance(r, (tuple, list)):
        return {"seq": [_encode(x, full) for x in r], "tuple": isinstance(r, tuple)}
    if isinstance(r, (bytes, np.ndarray)):
        raw = r if isinstance(r, bytes) else np.ascontiguousarray(r).tobytes()
        e = {"digest": _bytes_digest(raw)}
        if full:
            e["b64"] = base64.b64encode(raw).decode()
            if isinstance(r, np.ndarray):
                e["dtype"], e["shape"] = r.dtype.str, list(r.shape)
        return e
    return {"v": r.item() if isinstance(r, np.generic) else r}


def _decode(e):
    if "none" in e:
        return None
    if "seq" in e:
        s = [_decode(x) for x in e["seq"]]
        return tuple(s) if e["tuple"] else s
    if "digest" in e:
        if "b64" not in e:
            return Recorded(e["digest"])
        raw = base64.b64decode(e["b64"])
        return np.frombuffer(raw, dtype=e["dtype"]).reshape(e["shape"]).copy() if "dtype" in e else raw
    return e["v"]


def _store():
    global _recorded
    if _recorded is None:
        try:
            with open(_RECORDED_PATH) as f:
                _recorded = json.load(f)
        except FileNotFoundError:
            _recorded = {}
        if _record:
            atexit.register(_save)
    return _recorded


def _save():
    with open(_RECORDED_PATH, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, sort_keys=True)}" for k, v in sorted(_recorded.items())) + "\n}\n")


def _call_key(spec, name, args, kw):
    parts = [repr(spec), name]
    for a in list(args) + [kw[k] for k in sorted(kw)]:
        parts.append(_digest_of(a) if isinstance(a, (np.ndarray, bytes, Recorded)) else repr(a))
    return _bytes_digest("|".join(parts).encode())


def _replayed(spec, name, args, kw, live):
    """the live result (checked against, or with recording added to, the recorded one) or the recorded result"""
    store, key = _store(), _call_key(spec, name, args, kw)
    if live is None:
        if key not in store:
            raise KeyError(f"no recorded reference result for {name}{spec}; record it with SEAL_B200_RECORD_REFERENCE=1 where "
                           f"oracle/_ref is built")
        return _decode(store[key])
    r = live(*args, **kw)
    e = _encode(r, name in _DATA_METHODS)
    if key in store:
        assert store[key] == e, f"the live reference's {name}{spec} differs from {_RECORDED_PATH}"
    elif _record:
        store[key] = e
    return r


class Replay:
    """RefContext's methods, answered live when the reference library is built and from the recorded results otherwise"""

    def __init__(self, scheme, n, moduli, plain_modulus=0, seed=0x5EA1):
        self._spec = (scheme, n, [int(q) for q in moduli], int(plain_modulus), seed)
        self._live = RefContext(scheme, n, moduli, plain_modulus, seed) if available() else None

    def __getattr__(self, name):
        if name.startswith("_") or not callable(getattr(RefContext, name, None)):
            raise AttributeError(name)
        live = getattr(self._live, name) if self._live is not None else None
        return lambda *args, **kw: _replayed(self._spec, name, args, kw, live)


def replay(fn, *args):
    """one of this module's context-free functions (coeff_modulus_create, plain_modulus_batching, ...), live or recorded"""
    return _replayed((), fn.__name__, args, {}, fn if available() else None)


def coeff_modulus_create(n, bits):
    out = np.zeros(len(bits), dtype=np.uint64)
    b = (C.c_int * len(bits))(*bits)
    if lib().sealref_coeff_modulus_create(n, b, len(bits), _p(out)):
        raise RuntimeError(lib().sealref_last_error().decode())
    return [int(x) for x in out]


def coeff_modulus_bfv_default(n):
    out = np.zeros(64, dtype=np.uint64)
    k = C.c_size_t(0)
    if lib().sealref_coeff_modulus_bfv_default(n, _p(out), 64, C.byref(k)):
        raise RuntimeError(lib().sealref_last_error().decode())
    return [int(x) for x in out[: k.value]]


def plain_modulus_batching(n, bits):
    return int(lib().sealref_plain_modulus_batching(n, bits))


class RefContext:
    """One reference SEALContext + KeyGenerator + Evaluator (sec_level none, expand_mod_chain=true)."""

    def __init__(self, scheme, n, moduli, plain_modulus=0, seed=0x5EA1):
        self.scheme, self.n, self.moduli, self.k = scheme, n, list(moduli), len(moduli)
        self.plain_modulus = plain_modulus
        m = np.array(self.moduli, dtype=np.uint64)
        self.h = lib().sealref_create(scheme, n, _p(m), self.k, plain_modulus, seed)
        if not self.h:
            raise RuntimeError(lib().sealref_last_error().decode())

    def close(self):
        if self.h:
            lib().sealref_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError(lib().sealref_last_error().decode())

    def ntt_root(self, i):
        r = C.c_uint64(0)
        self._chk(lib().sealref_ntt_root(self.h, i, C.byref(r)))
        return r.value

    def ntt_tables(self, i):
        n = self.n
        a, b, c = (np.zeros(n, dtype=np.uint64) for _ in range(3))
        d = C.c_uint64(0)
        self._chk(lib().sealref_ntt_tables(self.h, i, _p(a), _p(b), _p(c), C.byref(d)))
        return a, b, c, d.value

    def base_bsk(self, L):
        out = np.zeros(self.k + 4, dtype=np.uint64)
        cnt = lib().sealref_base_bsk(self.h, L, _p(out), len(out))
        if cnt == 0:
            raise RuntimeError(lib().sealref_last_error().decode())
        return [int(x) for x in out[:cnt]]

    def relin_key(self):
        out = np.zeros((self.k - 1, 2, self.k, self.n), dtype=np.uint64)
        self._chk(lib().sealref_relin_key(self.h, _p(out)))
        return out

    def galois_key(self, elt):
        out = np.zeros((self.k - 1, 2, self.k, self.n), dtype=np.uint64)
        self._chk(lib().sealref_galois_key(self.h, elt, _p(out)))
        return out

    def galois_elt_from_step(self, step):
        return int(lib().sealref_galois_elt_from_step(self.h, step))

    def ntt_forward(self, L, data):
        d = np.ascontiguousarray(data).copy()
        self._chk(lib().sealref_ntt_forward(self.h, L, d.shape[0], _p(d)))
        return d

    def ntt_inverse(self, L, data):
        d = np.ascontiguousarray(data).copy()
        self._chk(lib().sealref_ntt_inverse(self.h, L, d.shape[0], _p(d)))
        return d

    def multiply(self, L, a, b):
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        sa, sb = a.shape[0], b.shape[0]
        out = np.zeros((sa + sb - 1, L, self.n), dtype=np.uint64)
        if (sa, sb) == (2, 2):
            self._chk(lib().sealref_multiply(self.h, L, _p(a), _p(b), _p(out)))
        else:
            self._chk(lib().sealref_multiply_sized(self.h, L, sa, sb, _p(a), _p(b), _p(out)))
        return out

    def square(self, L, a):
        out = np.zeros((3, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_square(self.h, L, _p(a), _p(out)))
        return out

    def linear(self, mode, L, a, b=None):
        a = np.ascontiguousarray(a)
        out = np.zeros_like(a)
        bb = np.ascontiguousarray(b) if b is not None else a
        self._chk(lib().sealref_linear(self.h, mode, L, a.shape[0], _p(a), _p(bb), _p(out)))
        return out

    def multiply_plain(self, L, a, plain):
        a, plain = np.ascontiguousarray(a), np.ascontiguousarray(plain)
        out = np.zeros_like(a)
        self._chk(lib().sealref_multiply_plain_ntt(self.h, L, a.shape[0], _p(a), _p(plain), _p(out)))
        return out

    def relinearize(self, L, c3):
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_relinearize(self.h, L, _p(c3), _p(out)))
        return out

    def multiply_relin(self, L, a, b):
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_multiply_relin(self.h, L, _p(a), _p(b), _p(out)))
        return out

    def rescale(self, L, c2):
        out = np.zeros((2, L - 1, self.n), dtype=np.uint64)
        self._chk(lib().sealref_rescale(self.h, L, _p(c2), _p(out)))
        return out

    def mod_switch(self, L, c2):
        out = np.zeros((2, L - 1, self.n), dtype=np.uint64)
        self._chk(lib().sealref_mod_switch(self.h, L, _p(c2), _p(out)))
        return out

    def apply_galois(self, L, c2, elt):
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_apply_galois(self.h, L, _p(c2), elt, _p(out)))
        return out

    def rotate(self, L, c2, step):
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_rotate(self.h, L, _p(c2), step, _p(out)))
        return out

    def bfv_encrypt(self, slots):
        out = np.zeros((2, self.k - 1, self.n), dtype=np.uint64)
        s = np.ascontiguousarray(slots, dtype=np.uint64)
        self._chk(lib().sealref_bfv_encrypt(self.h, _p(s), _p(out)))
        return out

    def bfv_decrypt(self, L, ct):
        ct = np.ascontiguousarray(ct)
        out = np.zeros(self.n, dtype=np.uint64)
        nb = C.c_int(0)
        self._chk(lib().sealref_bfv_decrypt(self.h, L, ct.shape[0], _p(ct), _p(out), C.byref(nb)))
        return out, nb.value

    def secret_key(self):
        out = np.zeros((self.k, self.n), dtype=np.uint64)
        self._chk(lib().sealref_secret_key(self.h, _p(out)))
        return out

    def decrypt(self, L, ct, is_ntt_form, correction_factor=1):
        """Decryptor::decrypt -> n words (BFV / BGV) or [L][n] (CKKS)"""
        ct = np.ascontiguousarray(ct)
        out = np.zeros((L, self.n) if self.scheme == CKKS else self.n, dtype=np.uint64)
        self._chk(lib().sealref_decrypt(self.h, L, ct.shape[0], int(is_ntt_form), correction_factor, _p(ct), _p(out)))
        return out

    def batch_codec(self, data, decode):
        data = np.ascontiguousarray(data, dtype=np.uint64)
        out = np.zeros(self.n, dtype=np.uint64)
        self._chk(lib().sealref_batch_codec(self.h, int(decode), _p(data), _p(out)))
        return out

    def plain_to_ntt(self, L, plain):
        plain = np.ascontiguousarray(plain, dtype=np.uint64)
        out = np.zeros((L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_plain_to_ntt(self.h, L, _p(plain), _p(out)))
        return out

    def plain_op_coeff(self, mode, L, a, plain, ct_is_ntt, correction_factor=1):
        """Evaluator.multiply_plain (0) / add_plain (1) / sub_plain (2) with a coefficient-form plaintext [n]"""
        a, plain = np.ascontiguousarray(a), np.ascontiguousarray(plain, dtype=np.uint64)
        out = np.zeros_like(a)
        self._chk(lib().sealref_plain_op_coeff(self.h, mode, L, a.shape[0], int(ct_is_ntt), correction_factor, _p(a), _p(plain), _p(out)))
        return out

    def parms_id(self, L):
        out = np.zeros(4, dtype=np.uint64)
        self._chk(lib().sealref_parms_id(self.h, L, _p(out)))
        return tuple(int(x) for x in out)

    def ct_save(self, L, data, is_ntt_form, scale=1.0, correction_factor=1, compr=0):
        """Ciphertext::save of [size][L][n] words with compr_mode none (0) or zlib (1)"""
        data = np.ascontiguousarray(data)
        buf = C.create_string_buffer(data.nbytes + data.nbytes // 8 + 4096)
        ln = lib().sealref_ct_save_mode(self.h, L, data.shape[0], _p(data), int(is_ntt_form), scale, correction_factor, compr, buf, len(buf))
        if ln < 0:
            raise RuntimeError(lib().sealref_last_error().decode())
        return buf.raw[:ln]

    def ct_load(self, stream, max_size=16):
        """Ciphertext::load -> (data [size][L][n], is_ntt_form, scale, correction_factor)"""
        out = np.zeros(max_size * self.k * self.n, dtype=np.uint64)
        size, L, cf = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        ntt, scale = C.c_int(0), C.c_double(0)
        self._chk(lib().sealref_ct_load(self.h, stream, len(stream), _p(out), out.size, C.byref(size), C.byref(L), C.byref(ntt),
                                        C.byref(scale), C.byref(cf)))
        return out[: size.value * L.value * self.n].reshape(size.value, L.value, self.n).copy(), bool(ntt.value), scale.value, cf.value

    def kswitch_keys_stream(self, galois_elt=0, compr=0):
        """RelinKeys::save (galois_elt == 0) or GaloisKeys::save of the keys holding that element, compr_mode none (0) / zlib (1)"""
        raw = (self.k - 1) * 2 * self.k * self.n * 8
        buf = C.create_string_buffer(raw + raw // 8 + 8 * self.n + (1 << 16))
        ln = lib().sealref_kswitch_keys_stream_mode(self.h, galois_elt, compr, buf, len(buf))
        if ln < 0:
            raise RuntimeError(lib().sealref_last_error().decode())
        return buf.raw[:ln]

    def ckks_encode(self, L, values, scale):
        """CKKSEncoder::encode(vector<complex<double>>, parms_id of level L, scale) -> [L][n] (NTT form), or None when the
        reference throws invalid_argument"""
        v = np.ascontiguousarray(values, dtype=np.complex128)
        out = np.zeros((L, self.n), dtype=np.uint64)
        rc = lib().sealref_ckks_encode(self.h, L, v.ctypes.data, v.size, float(scale), _p(out))
        if rc == 1:
            return None
        self._chk(rc)
        return out

    def ckks_decode(self, L, plain, scale):
        """CKKSEncoder::decode -> n/2 complex values, or None when the reference throws invalid_argument"""
        plain = np.ascontiguousarray(plain, dtype=np.uint64)
        out = np.zeros(self.n // 2, dtype=np.complex128)
        rc = lib().sealref_ckks_decode(self.h, L, _p(plain), float(scale), out.ctypes.data)
        if rc == 1:
            return None
        self._chk(rc)
        return out

    def public_key(self):
        """KeyGenerator::create_public_key -> [2][k][n] (NTT form, key level)"""
        out = np.zeros((2, self.k, self.n), dtype=np.uint64)
        self._chk(lib().sealref_public_key(self.h, _p(out)))
        return out

    def encrypt_zero_asymmetric(self, L=None):
        """Encryptor(public key)::encrypt_zero(parms_id of the level with L primes; L == k: the key level) -> [2][L][n]"""
        L = L or (self.k - 1 if self.k > 1 else 1)
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_encrypt_zero_asymmetric(self.h, L, _p(out)))
        return out

    def encrypt_zero_symmetric(self, L=None):
        """Encryptor::encrypt_zero_symmetric(parms_id, ct) (not seed-compressed) -> [2][L][n]; the bootstrap PRNG is seeded with
        {seed, 0, ...} (deterministic)"""
        L = L or (self.k - 1 if self.k > 1 else 1)
        out = np.zeros((2, L, self.n), dtype=np.uint64)
        self._chk(lib().sealref_encrypt_zero_symmetric(self.h, L, _p(out)))
        return out

    def seeded_ct_stream(self, compr=0):
        buf = C.create_string_buffer(2 * self.k * self.n * 8 + self.k * self.n + 4096)
        ln = lib().sealref_seeded_ct_stream_mode(self.h, compr, buf, len(buf))
        if ln < 0:
            raise RuntimeError(lib().sealref_last_error().decode())
        return buf.raw[:ln]

    def time_op(self, op, L, threads, reps):
        t = lib().sealref_time_op(self.h, op, L, threads, reps)
        if t < 0:
            raise RuntimeError(lib().sealref_last_error().decode())
        return t
