"""Device and host-buffer entry points of every evaluator operation (-m gpu).  For each operation of include/seal_b200.h the
sb200_X / sb200_X_host pair must compute the same words, reject the same invalid arguments with the same status, move
per-ciphertext correction factors along with the staging chunks, and follow the aliasing rule of the host variants: in several
chunks the output may overlap an input only exactly in place with an output no larger than that input.  Host calls run in
staging chunks of 2 ciphertexts (2, 2, 2, 1 for a batch of 7) unless a test says otherwise."""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from common import rand_ct

pytestmark = pytest.mark.gpu

N, K, L, BATCH, CHUNK = 4096, 4, 3, 7, 2
E_INVALID_ARG = -1
OUT = "out"
sz, i32, u32 = C.c_size_t, C.c_int, C.c_uint32
SCHEMES = {"bfv": 1, "ckks": 2, "bgv": 3}
COMMON = ["ntt_forward", "ntt_inverse", "multiply", "multiply_sized", "square", "add", "sub", "negate", "relinearize", "relinearize_sized",
          "multiply_relinearize", "mod_switch_to_next", "mod_switch_to_next_sized", "apply_galois", "decrypt"]
COEFF = ["plain_to_ntt", "multiply_plain_coeff", "add_plain_coeff", "batch_encode", "batch_decode"]
NAMES = {"ckks": COMMON + ["rescale_to_next", "rescale_to_next_sized", "multiply_plain"], "bfv": COMMON + COEFF,
         "bgv": COMMON + COEFF + ["multiply_plain"]}
SIZED = {"multiply_sized", "relinearize_sized", "rescale_to_next_sized", "mod_switch_to_next_sized"}
CASES = [(s, name) for s in SCHEMES for name in NAMES[s]]


class In:
    """input i of a call (OUT: its output)"""

    def __init__(self, i):
        self.i = i


class Env:
    """a small context of one scheme (n = 4096, k = 4) with a relinearization key, a Galois key and a secret key of random words"""

    def __init__(self, scheme):
        import seal_b200

        self.scheme = scheme
        self.mods = O.coeff_modulus_create(N, [50] * K)
        self.t = 0 if scheme == seal_b200.CKKS else next(p for p in range((1 << 20) + 1, 1 << 21, 2 * N) if O.lib().orc_is_prime(p))
        self.ctx = seal_b200.Context(scheme, N, self.mods, self.t)
        rng = np.random.default_rng(100 + scheme)
        self.relin = self.ctx.load_key(rng.integers(0, 1 << 40, (K - 1, 2, K, N), dtype=np.uint64))
        self.galois = self.ctx.load_key(rng.integers(0, 1 << 40, (K - 1, 2, K, N), dtype=np.uint64))
        self.sk = self.ctx.load_secret_key(rng.integers(0, 1 << 40, (K, N), dtype=np.uint64))
        self.cf = rng.integers(1, max(self.t, 2), BATCH, dtype=np.uint64)  # BGV correction factors, invertible mod t
        self.lib = C.CDLL(seal_b200.LIB_PATH)  # a handle without argtypes: every argument is an explicit ctypes value
        self.lib.sb200_last_error.restype = C.c_char_p

    def ct(self, size, seed):
        return rand_ct(np.random.default_rng(seed), self.mods, N, size, L, BATCH)

    def plain(self, seed):
        return np.random.default_rng(seed).integers(0, self.t, (BATCH, N), dtype=np.uint64)

    def stage_limit(self, value):
        assert self.lib.sb200_context_set_limit(self.ctx.h, i32(self.ctx.LIMIT_HOST_STAGE_BYTES), sz(value)) == 0

    def operations(self):
        """name -> (args(level, batch, size), inputs, output): the arguments after the context, In(i) / OUT for the buffers"""
        bgv, ckks = self.scheme == 3, self.scheme == 2
        cf = C.c_void_p(self.cf.ctypes.data) if bgv else C.c_void_p(None)
        z = lambda *shape: np.zeros((BATCH,) + shape, np.uint64)  # noqa: E731
        ops = {
            "ntt_forward": (lambda l, b, s=None: [sz(l), sz(2), sz(b), OUT], [], self.ct(2, 1)),
            "ntt_inverse": (lambda l, b, s=None: [sz(l), sz(2), sz(b), OUT], [], self.ct(2, 2)),
            "multiply": (lambda l, b, s=None: [sz(l), sz(b), In(0), In(1), OUT], [self.ct(2, 3), self.ct(2, 4)], z(3, L, N)),
            "multiply_sized": (lambda l, b, s=3: [sz(l), sz(s), sz(2), sz(b), In(0), In(1), OUT], [self.ct(3, 5), self.ct(2, 6)], z(4, L, N)),
            "square": (lambda l, b, s=None: [sz(l), sz(b), In(0), OUT], [self.ct(2, 7)], z(3, L, N)),
            "add": (lambda l, b, s=None: [sz(l), sz(2), sz(b), In(0), In(1), OUT], [self.ct(2, 8), self.ct(2, 9)], z(2, L, N)),
            "sub": (lambda l, b, s=None: [sz(l), sz(2), sz(b), In(0), In(1), OUT], [self.ct(2, 10), self.ct(2, 11)], z(2, L, N)),
            "negate": (lambda l, b, s=None: [sz(l), sz(2), sz(b), In(0), OUT], [self.ct(2, 12)], z(2, L, N)),
            "relinearize": (lambda l, b, s=None: [sz(l), sz(b), In(0), self.relin.h, OUT], [self.ct(3, 13)], z(2, L, N)),
            "relinearize_sized": (lambda l, b, s=4: [sz(l), sz(s), sz(b), In(0), self.relin.h, OUT], [self.ct(4, 14)], z(4, L, N)),
            "multiply_relinearize": (lambda l, b, s=None: [sz(l), sz(b), In(0), In(1), self.relin.h, OUT], [self.ct(2, 15), self.ct(2, 16)],
                                     z(2, L, N)),
            "mod_switch_to_next": (lambda l, b, s=None: [sz(l), sz(b), In(0), OUT], [self.ct(2, 17)], z(2, L - 1, N)),
            "mod_switch_to_next_sized": (lambda l, b, s=3: [sz(l), sz(s), sz(b), In(0), OUT], [self.ct(3, 18)], z(3, L - 1, N)),
            "apply_galois": (lambda l, b, s=None: [sz(l), sz(b), In(0), u32(3), self.galois.h, OUT], [self.ct(2, 19)], z(2, L, N)),
            "decrypt": (lambda l, b, s=None: [self.sk.h, sz(l), sz(2), sz(b), In(0), cf, OUT], [self.ct(2, 20)], z(L, N) if ckks else z(N)),
            "rescale_to_next": (lambda l, b, s=None: [sz(l), sz(b), In(0), OUT], [self.ct(2, 21)], z(2, L - 1, N)),
            "rescale_to_next_sized": (lambda l, b, s=3: [sz(l), sz(s), sz(b), In(0), OUT], [self.ct(3, 22)], z(3, L - 1, N)),
            "multiply_plain": (lambda l, b, s=None: [sz(l), sz(2), sz(b), In(0), In(1), OUT], [self.ct(2, 23), self.ct(1, 24)[:, 0]], z(2, L, N)),
        }
        if not ckks:
            ops.update({
                "plain_to_ntt": (lambda l, b, s=None: [sz(l), sz(b), In(0), OUT], [self.plain(25)], z(L, N)),
                "multiply_plain_coeff": (lambda l, b, s=None: [sz(l), sz(2), sz(b), i32(1 if bgv else 0), In(0), In(1), OUT],
                                         [self.ct(2, 26), self.plain(27)], z(2, L, N)),
                "add_plain_coeff": (lambda l, b, s=None: [sz(l), sz(2), sz(b), i32(0), In(0), In(1), cf, OUT], [self.ct(2, 28), self.plain(29)],
                                    z(2, L, N)),
                "batch_encode": (lambda l, b, s=None: [sz(b), In(0), OUT], [self.plain(30)], z(N)),
                "batch_decode": (lambda l, b, s=None: [sz(b), In(0), OUT], [self.plain(31)], z(N)),
            })
        return ops

    def multi_chunk(self, ins, out):
        """stage limit that cuts BATCH ciphertexts of an operation with these buffers into chunks of CHUNK"""
        self.stage_limit(CHUNK * sum(x.size for x in ins + [out]) // BATCH * 8)

    def invoke(self, name, args, ins, out, device):
        """sb200_<name> (device slabs, current stream) or sb200_<name>_host on copies of `ins` and `out`.
        Returns (status, message, [inputs..., output]) with the buffers as they are after the call."""
        import torch

        if device:
            bufs = [torch.from_numpy(np.ascontiguousarray(x).copy().view(np.int64)).cuda() for x in ins + [out]]
            ptr = [C.c_void_p(b.data_ptr()) for b in bufs]
        else:
            bufs = [np.ascontiguousarray(x).copy() for x in ins + [out]]
            ptr = [C.c_void_p(b.ctypes.data) for b in bufs]
        cargs = [ptr[a.i] if isinstance(a, In) else ptr[-1] if a is OUT else a for a in args]
        if device:
            cargs.append(C.c_void_p(torch.cuda.current_stream().cuda_stream))
        rc = getattr(self.lib, "sb200_" + name + ("" if device else "_host"))(self.ctx.h, *cargs)
        msg = self.lib.sb200_last_error().decode()
        if device:
            torch.cuda.synchronize()
            bufs = [b.cpu().numpy().view(np.uint64) for b in bufs]
        return rc, msg, bufs


_envs = {}


def env(scheme):
    if scheme not in _envs:
        _envs[scheme] = Env(SCHEMES[scheme])
        _envs[scheme].ops = _envs[scheme].operations()
    return _envs[scheme]


def aliased(args, j):
    """the same call with the output written over input j"""
    return [In(j) if a is OUT else a for a in args]


@pytest.mark.parametrize("scheme,name", CASES)
def test_device_equals_host(scheme, name):
    e = env(scheme)
    args, ins, out = e.ops[name]
    e.multi_chunk(ins, out)
    try:
        rc_d, msg_d, dev = e.invoke(name, args(L, BATCH), ins, out, True)
        rc_h, msg_h, host = e.invoke(name, args(L, BATCH), ins, out, False)
    finally:
        e.stage_limit(640 << 20)
    assert rc_d == 0, msg_d
    assert rc_h == 0, msg_h
    assert (dev[-1] == host[-1]).all(), "device and host outputs differ"
    assert (host[-1] != out).any(), "the output was not written"


@pytest.mark.parametrize("scheme,name", CASES)
def test_invalid_arguments(scheme, name):
    e = env(scheme)
    args, ins, out = e.ops[name]
    calls = [args(L, 0)]  # batch = 0
    if not name.startswith("batch_"):
        calls += [args(0, BATCH), args(K + 1, BATCH)]
    if name in SIZED:
        calls += [args(L, BATCH, 0), args(L, BATCH, 17)]
    if name.startswith(("rescale", "mod_switch")):
        calls.append(args(1, BATCH))
    e.multi_chunk(ins, out)
    try:
        for c in calls:
            for device in (True, False):
                rc, msg, bufs = e.invoke(name, c, ins, out, device)
                assert rc == E_INVALID_ARG, (device, msg)
                assert (bufs[-1] == out).all(), "a rejected call wrote its output"
        # device slabs of these operations change layout: aliasing is rejected
        alias = {"multiply_sized": [0, 1], "relinearize": [0], "relinearize_sized": [0], "apply_galois": [0], "rescale_to_next": [0],
                 "rescale_to_next_sized": [0], "mod_switch_to_next": [0], "mod_switch_to_next_sized": [0]}.get(name, [])
        for j in alias:
            rc, msg, _ = e.invoke(name, aliased(args(L, BATCH), j), ins, out, True)
            assert rc == E_INVALID_ARG, msg
    finally:
        e.stage_limit(640 << 20)


@pytest.mark.parametrize("name", ["add_plain_coeff", "decrypt"])
def test_correction_factors_move_with_the_chunks(name):
    """BGV: per-ciphertext correction factors in a multi-chunk host call and a device call equal one call per ciphertext"""
    e = env("bgv")
    args, ins, out = e.ops[name]
    singles = []
    for i in range(BATCH):
        one = [C.c_void_p(e.cf[i:].ctypes.data) if isinstance(a, C.c_void_p) and a.value == e.cf.ctypes.data else a for a in args(L, 1)]
        rc, msg, bufs = e.invoke(name, one, [x[i:i + 1] for x in ins], out[i:i + 1], False)
        assert rc == 0, msg
        singles.append(bufs[-1][0])
    e.multi_chunk(ins, out)
    try:
        for device in (True, False):
            rc, msg, bufs = e.invoke(name, args(L, BATCH), ins, out, device)
            assert rc == 0, msg
            assert (bufs[-1] == np.stack(singles)).all(), f"device={device}: correction factors did not follow the ciphertexts"
    finally:
        e.stage_limit(640 << 20)


IN_PLACE = [("ckks", "add"), ("ckks", "sub"), ("ckks", "negate"), ("ckks", "multiply_plain"), ("ckks", "relinearize"), ("ckks", "apply_galois"),
            ("ckks", "rescale_to_next"), ("bgv", "multiply_plain")]


@pytest.mark.parametrize("scheme,name", IN_PLACE)
def test_host_in_place_no_larger_output(scheme, name):
    """h_out == h_a with an output no larger than the input: the multi-chunk host call equals the out-of-place one"""
    e = env(scheme)
    args, ins, out = e.ops[name]
    e.multi_chunk(ins, out)
    try:
        rc, msg, want = e.invoke(name, args(L, BATCH), ins, out, False)
        assert rc == 0, msg
        rc, msg, got = e.invoke(name, aliased(args(L, BATCH), 0), ins, out, False)
        assert rc == 0, msg
    finally:
        e.stage_limit(640 << 20)
    assert (got[0].reshape(-1)[: out.size] == want[-1].reshape(-1)).all()


GROWING = [("ckks", "multiply"), ("ckks", "square"), ("ckks", "multiply_sized"), ("bgv", "plain_to_ntt")]


@pytest.mark.parametrize("scheme,name", GROWING)
def test_host_in_place_larger_output(scheme, name):
    """h_out == h_a with an output larger than the input: refused in several chunks (a chunk's output would overwrite input
    rows of a later chunk), computed as out of place in one chunk"""
    e = env(scheme)
    args, ins, out = e.ops[name]
    buf = np.zeros(out.size, np.uint64)
    buf[: ins[0].size] = ins[0].reshape(-1)
    e.multi_chunk(ins, out)
    try:
        rc, msg, got = e.invoke(name, aliased(args(L, BATCH), 0), [buf] + ins[1:], out, False)
    finally:
        e.stage_limit(640 << 20)
    assert rc == E_INVALID_ARG, "multi-chunk call with a growing in-place output was accepted"
    assert (got[0] == buf).all(), "a refused call changed the buffer"
    # a batch of 3 fits one staging chunk
    B = 3
    small = [x[:B] for x in ins]
    rc, msg, want = e.invoke(name, args(L, B), small, out[:B], False)
    assert rc == 0, msg
    buf = np.zeros(out[:B].size, np.uint64)
    buf[: small[0].size] = small[0].reshape(-1)
    rc, msg, got = e.invoke(name, aliased(args(L, B), 0), [buf] + small[1:], out[:B], False)
    assert rc == 0, msg
    assert (got[0] == want[-1].reshape(-1)).all()


def test_host_multiply_sized_into_second_operand():
    """Evaluator::multiply_inplace(x, y) of the C++ shim: one ciphertext, the product written over the second operand"""
    e = env("ckks")
    args, ins, out = e.ops["multiply_sized"]
    small = [x[:1] for x in ins]
    rc, msg, want = e.invoke("multiply_sized", args(L, 1), small, out[:1], False)
    assert rc == 0, msg
    buf = np.zeros(out[:1].size, np.uint64)
    buf[: small[1].size] = small[1].reshape(-1)
    rc, msg, got = e.invoke("multiply_sized", aliased(args(L, 1), 1), [small[0], buf], out[:1], False)
    assert rc == 0, msg
    assert (got[1] == want[-1].reshape(-1)).all()
