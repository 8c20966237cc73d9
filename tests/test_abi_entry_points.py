"""CPU test: the argument checks that run before a context is touched, for the device and host-buffer entry points of every
evaluator operation in include/seal_b200.h.  Each entry point is called once with a null context and every other pointer valid,
and once with every pointer null; the status code and sb200_last_error() must match the table below.  The table pins which
pointer each entry point checks first.  No call passes a context, so nothing here needs a GPU."""
import ctypes as C

import pytest

# argument kinds in declaration order: c = context, p = pointer, n = size_t, i = int, u = uint32, s = stream (may be NULL).
# The host-buffer variant of each operation takes the same arguments without the stream.
DEVICE_SIGNATURES = {
    "sb200_ntt_forward": "cnnnps",
    "sb200_ntt_inverse": "cnnnps",
    "sb200_multiply": "cnnppps",
    "sb200_multiply_sized": "cnnnnppps",
    "sb200_square": "cnnpps",
    "sb200_add": "cnnnppps",
    "sb200_sub": "cnnnppps",
    "sb200_negate": "cnnnpps",
    "sb200_multiply_plain": "cnnnppps",
    "sb200_plain_to_ntt": "cnnpps",
    "sb200_multiply_plain_coeff": "cnnnippps",
    "sb200_add_plain_coeff": "cnnnipppps",
    "sb200_batch_encode": "cnpps",
    "sb200_batch_decode": "cnpps",
    "sb200_relinearize": "cnnppps",
    "sb200_relinearize_sized": "cnnnppps",
    "sb200_multiply_relinearize": "cnnpppps",
    "sb200_rescale_to_next": "cnnpps",
    "sb200_rescale_to_next_sized": "cnnnpps",
    "sb200_mod_switch_to_next": "cnnpps",
    "sb200_mod_switch_to_next_sized": "cnnnpps",
    "sb200_apply_galois": "cnnpupps",
    "sb200_decrypt": "cpnnnppps",
}
SIGNATURES = dict(DEVICE_SIGNATURES)
SIGNATURES.update({name + "_host": kinds[:-1] for name, kinds in DEVICE_SIGNATURES.items()})

# (status, message) with a null context and every other pointer valid; (status, message) with every pointer null
EXPECTED = {
    "sb200_add": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_add_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_add_plain_coeff": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_add_plain_coeff_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_apply_galois": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_apply_galois_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_batch_decode": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_batch_decode_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_batch_encode": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_batch_encode_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_decrypt": ((-6, "null pointer: ctx"), (-6, "null pointer: key")),
    "sb200_decrypt_host": ((-6, "null pointer: ctx"), (-6, "null pointer: key")),
    "sb200_mod_switch_to_next": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_mod_switch_to_next_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_mod_switch_to_next_sized": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_mod_switch_to_next_sized_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_multiply": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_plain": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_plain_coeff": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_plain_coeff_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_plain_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_relinearize": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_relinearize_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_sized": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_multiply_sized_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_negate": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_negate_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_ntt_forward": ((-6, "null pointer: ctx"), (-6, "null pointer: d")),
    "sb200_ntt_forward_host": ((-6, "null pointer: ctx"), (-6, "null pointer: h")),
    "sb200_ntt_inverse": ((-6, "null pointer: ctx"), (-6, "null pointer: d")),
    "sb200_ntt_inverse_host": ((-6, "null pointer: ctx"), (-6, "null pointer: h")),
    "sb200_plain_to_ntt": ((-6, "null pointer: ctx"), (-6, "null pointer: plain")),
    "sb200_plain_to_ntt_host": ((-6, "null pointer: ctx"), (-6, "null pointer: plain")),
    "sb200_relinearize": ((-6, "null pointer: ctx"), (-6, "null pointer: in3")),
    "sb200_relinearize_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in3")),
    "sb200_relinearize_sized": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_relinearize_sized_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_rescale_to_next": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_rescale_to_next_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_rescale_to_next_sized": ((-6, "null pointer: ctx"), (-6, "null pointer: in")),
    "sb200_rescale_to_next_sized_host": ((-6, "null pointer: ctx"), (-6, "null pointer: in2")),
    "sb200_square": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_square_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_sub": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
    "sb200_sub_host": ((-6, "null pointer: ctx"), (-6, "null pointer: a")),
}


def _lib():
    import seal_b200

    seal_b200.lib()  # fails loudly when the library has not been built
    lib = C.CDLL(seal_b200.LIB_PATH)  # a handle of its own: no argtypes, every argument is passed as an explicit ctypes value
    lib.sb200_last_error.restype = C.c_char_p
    return lib


def _call(lib, name, null_ctx_only):
    bufs = []
    args = []
    for kind in SIGNATURES[name]:
        if kind == "c":
            args.append(C.c_void_p(None))
        elif kind in "ps":
            if null_ctx_only and kind == "p":
                bufs.append(C.create_string_buffer(64))  # distinct buffers: no alias check can fire first
                args.append(C.cast(bufs[-1], C.c_void_p))
            else:
                args.append(C.c_void_p(None))
        elif kind == "n":
            args.append(C.c_size_t(2))
        elif kind == "i":
            args.append(C.c_int(0))
        elif kind == "u":
            args.append(C.c_uint32(3))
    rc = getattr(lib, name)(*args)
    return rc, lib.sb200_last_error().decode()


def observed():
    lib = _lib()
    return {name: (_call(lib, name, True), _call(lib, name, False)) for name in sorted(SIGNATURES)}


def test_table_covers_every_pair():
    assert len(SIGNATURES) == 2 * 23
    assert sorted(EXPECTED) == sorted(SIGNATURES)


@pytest.mark.parametrize("name", sorted(SIGNATURES))
def test_null_arguments(name):
    lib = _lib()
    null_ctx, all_null = EXPECTED[name]
    assert _call(lib, name, True) == tuple(null_ctx), "null context, every other pointer valid"
    assert _call(lib, name, False) == tuple(all_null), "every pointer null"
