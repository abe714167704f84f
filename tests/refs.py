"""ctypes access to the CPU oracle (oracle/_build/liboracle.so), to the answers of the unmodified reference
stored under tests/golden, and, when it was built, to the reference itself (oracle/_ref/*.so).  Test
infrastructure only."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libbz3_ref.so")
REF_STAGES_SO = os.path.join(ROOT, "oracle", "_ref", "libbz3_ref_stages.so")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "bzip3_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")
ANSWERS = os.path.join(GOLDEN, "reference_answers.json")

u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)


def digest(b) -> str:
    """Content digest of a byte string in the stored reference answers: the first 16 hex digits of its SHA-256."""
    return hashlib.sha256(bytes(b)).hexdigest()[:16]


_answers = None


def reference_answer(key):
    """What the unmodified reference computed for `key`, as written by tests/golden/make_reference_answers.py."""
    global _answers
    if _answers is None:
        with open(ANSWERS) as f:
            _answers = json.load(f)
    return _answers[key]


def check_answer(key, got):
    """`got` (ints, strings and lists of them) must equal the stored reference answer for `key`."""
    got, want = json.loads(json.dumps(got)), reference_answer(key)
    assert got == want, f"{key}: {got} differs from the reference's {want}"


def build_oracle():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
            os.path.join(ROOT, "oracle", "bz3_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "_build/liboracle.so"])


def ptr(a):
    return a.ctypes.data_as(u8p)


def bound(n):
    return n + n // 50 + 32


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        build_oracle()
        L = C.CDLL(ORACLE_SO)
        L.orc_crc32.restype = C.c_uint32
        L.orc_crc32.argtypes = [C.c_uint32, u8p, C.c_size_t]
        L.orc_mrle_encode.restype = C.c_int32
        L.orc_mrle_encode.argtypes = [u8p, C.c_int32, u8p]
        L.orc_mrle_decode.restype = C.c_int
        L.orc_mrle_decode.argtypes = [u8p, u8p, C.c_int32, C.c_int32]
        L.orc_lzp_encode.restype = C.c_int32
        L.orc_lzp_encode.argtypes = [u8p, C.c_int32, u8p, i32p]
        L.orc_lzp_decode.restype = C.c_int32
        L.orc_lzp_decode.argtypes = [u8p, C.c_int32, u8p, C.c_int32, i32p]
        L.orc_bwt.restype = C.c_int32
        L.orc_bwt.argtypes = [u8p, u8p, C.c_int32]
        L.orc_unbwt.restype = C.c_int32
        L.orc_unbwt.argtypes = [u8p, u8p, C.c_int32, C.c_int32]
        L.orc_cm_encode.restype = C.c_int32
        L.orc_cm_encode.argtypes = [u8p, C.c_int32, u8p]
        L.orc_cm_decode.restype = C.c_int32
        L.orc_cm_decode.argtypes = [u8p, C.c_int32, u8p, C.c_int32]
        L.orc_encode_block.restype = C.c_int32
        L.orc_encode_block.argtypes = [C.c_int32, u8p, C.c_int32, C.POINTER(C.c_int8)]
        L.orc_decode_block.restype = C.c_int32
        L.orc_decode_block.argtypes = [C.c_int32, u8p, C.c_size_t, C.c_int32, C.c_int32, C.POINTER(C.c_int8)]
        _oracle = L
    return _oracle


def have_ref():
    return os.path.exists(REF_SO) and os.path.exists(REF_STAGES_SO)


def declare_bz3_api(L):
    """Declare the libbz3.h prototypes on a loaded library (reference or ours: same ABI)."""
    L.bz3_version.restype = C.c_char_p
    L.bz3_new.restype = C.c_void_p
    L.bz3_new.argtypes = [C.c_int32]
    L.bz3_free.argtypes = [C.c_void_p]
    L.bz3_last_error.restype = C.c_int8
    L.bz3_last_error.argtypes = [C.c_void_p]
    L.bz3_strerror.restype = C.c_char_p
    L.bz3_strerror.argtypes = [C.c_void_p]
    L.bz3_bound.restype = C.c_size_t
    L.bz3_bound.argtypes = [C.c_size_t]
    L.bz3_encode_block.restype = C.c_int32
    L.bz3_encode_block.argtypes = [C.c_void_p, u8p, C.c_int32]
    L.bz3_decode_block.restype = C.c_int32
    L.bz3_decode_block.argtypes = [C.c_void_p, u8p, C.c_size_t, C.c_int32, C.c_int32]
    L.bz3_encode_blocks.restype = None
    L.bz3_encode_blocks.argtypes = [C.POINTER(C.c_void_p), C.POINTER(u8p), i32p, C.c_int32]
    L.bz3_decode_blocks.restype = None
    L.bz3_decode_blocks.argtypes = [C.POINTER(C.c_void_p), C.POINTER(u8p), C.POINTER(C.c_size_t), i32p, i32p,
                                    C.c_int32]
    L.bz3_compress.restype = C.c_int
    L.bz3_compress.argtypes = [C.c_uint32, u8p, u8p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.bz3_decompress.restype = C.c_int
    L.bz3_decompress.argtypes = [u8p, u8p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.bz3_min_memory_needed.restype = C.c_size_t
    L.bz3_min_memory_needed.argtypes = [C.c_int32]
    L.bz3_orig_size_sufficient_for_decode.restype = C.c_int
    L.bz3_orig_size_sufficient_for_decode.argtypes = [u8p, C.c_size_t, C.c_int32]
    return L


_ref = None
_ref_stages = None


def ref():
    global _ref
    if _ref is None:
        _ref = declare_bz3_api(C.CDLL(REF_SO))
    return _ref


def ref_stages():
    global _ref_stages
    if _ref_stages is None:
        L = C.CDLL(REF_STAGES_SO)
        L.ref_crc32.restype = C.c_uint32
        L.ref_crc32.argtypes = [C.c_uint32, u8p, C.c_size_t]
        L.ref_mrlec.restype = C.c_int32
        L.ref_mrlec.argtypes = [u8p, C.c_int32, u8p]
        L.ref_mrled.restype = C.c_int
        L.ref_mrled.argtypes = [u8p, u8p, C.c_int32, C.c_int32]
        L.ref_lzp_compress.restype = C.c_int32
        L.ref_lzp_compress.argtypes = [u8p, u8p, C.c_int32, i32p]
        L.ref_lzp_decompress.restype = C.c_int32
        L.ref_lzp_decompress.argtypes = [u8p, u8p, C.c_int32, C.c_int32, i32p]
        L.ref_bwt.restype = C.c_int32
        L.ref_bwt.argtypes = [u8p, u8p, i32p, C.c_int32]
        L.ref_unbwt.restype = C.c_int32
        L.ref_unbwt.argtypes = [u8p, u8p, i32p, C.c_int32, C.c_int32]
        L.ref_cm_encode.restype = C.c_int32
        L.ref_cm_encode.argtypes = [u8p, C.c_int32, u8p]
        L.ref_cm_decode.restype = None
        L.ref_cm_decode.argtypes = [u8p, C.c_int32, u8p, C.c_int32]
        _ref_stages = L
    return _ref_stages


# ---------------------------------------------------------------- block helpers
def api_encode_block(L, data: bytes, block_size: int):
    """Returns (encoded bytes or None, return value, last_error) through a libbz3-ABI library."""
    st = L.bz3_new(block_size)
    assert st, "bz3_new failed"
    try:
        n = len(data)
        buf = np.zeros(bound(max(n, block_size)) + 64, dtype=np.uint8)
        buf[:n] = np.frombuffer(data, dtype=np.uint8)
        r = L.bz3_encode_block(st, ptr(buf), n)
        e = L.bz3_last_error(st)
        return (bytes(buf[:r]) if r >= 0 else None), r, e
    finally:
        L.bz3_free(st)


def api_decode_block(L, enc: bytes, orig_size: int, block_size: int, buffer_size=None, compressed_size=None):
    st = L.bz3_new(block_size)
    assert st
    try:
        cap = bound(block_size) + 64
        buf = np.zeros(max(cap, len(enc)), dtype=np.uint8)
        buf[:len(enc)] = np.frombuffer(enc, dtype=np.uint8)
        bs = cap if buffer_size is None else buffer_size
        cs = len(enc) if compressed_size is None else compressed_size
        r = L.bz3_decode_block(st, ptr(buf), bs, cs, orig_size)
        e = L.bz3_last_error(st)
        return (bytes(buf[:r]) if r >= 0 else None), r, e
    finally:
        L.bz3_free(st)


def oracle_encode_block(data: bytes, block_size: int, err_init=0):
    O = oracle()
    n = len(data)
    buf = np.zeros(bound(max(n, block_size)) + 64, dtype=np.uint8)
    buf[:n] = np.frombuffer(data, dtype=np.uint8)
    err = C.c_int8(err_init)
    r = O.orc_encode_block(block_size, ptr(buf), n, C.byref(err))
    return (bytes(buf[:r]) if r >= 0 else None), r, err.value


def oracle_decode_block(enc: bytes, orig_size: int, block_size: int, buffer_size=None, compressed_size=None,
                        err_init=0):
    O = oracle()
    cap = bound(block_size) + 64
    buf = np.zeros(max(cap, len(enc)), dtype=np.uint8)
    buf[:len(enc)] = np.frombuffer(enc, dtype=np.uint8)
    bs = cap if buffer_size is None else buffer_size
    cs = len(enc) if compressed_size is None else compressed_size
    err = C.c_int8(err_init)
    r = O.orc_decode_block(block_size, ptr(buf), bs, cs, orig_size, C.byref(err))
    return (bytes(buf[:r]) if r >= 0 else None), r, err.value
