"""ORACLE — TEST INFRASTRUCTURE ONLY. ctypes binding of oracle/_build/libkanzi_oracle.so.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
It is the checker (a C++ restatement of kanzi-go's per-block path, see oracle/kzo.hpp), never the product.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libkanzi_oracle.so")

E_NONE, E_HUFFMAN, E_RANGE, E_ANS0, E_ANS1 = 0, 1, 4, 5, 8
T_NONE, T_BWT, T_BWTS, T_LZ, T_ROLZ, T_LZX = 0, 1, 2, 3, 11, 16
T_ZRLT, T_MTFT, T_RANK = 6, 7, 8
T_TEXT, T_MM, T_UTF, T_PACK, T_DNA, T_EXE = 10, 15, 17, 18, 19, 9  # oracle only so far (SURVEY.md 8(f) rank 2)


def build(force=False):
    # the TEXT codec's static dictionary is a format constant of the reference: written from tests/golden/ into oracle/_ref/ (not committed)
    from . import gen_text_dict

    gen_text_dict.main()
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp"))]
    srcs.append(gen_text_dict.OUT)
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs if os.path.exists(s)):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        u8p = C.POINTER(C.c_uint8)
        L.kzo_last_error.restype = C.c_char_p
        L.kzo_entropy_encode.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.kzo_entropy_decode.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.kzo_transform_forward.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        L.kzo_transform_inverse.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.kzo_set_stream_block_size.argtypes = [C.c_size_t]
        L.kzo_set_stream_block_size.restype = None
        L.kzo_transform_max_encoded_len.argtypes = [C.c_uint64, C.c_size_t]
        L.kzo_transform_max_encoded_len.restype = C.c_size_t
        L.kzo_bwt_forward_raw.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.kzo_bwt_forward_raw.restype = None
        L.kzo_bwt_inverse_raw.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.kzo_encode_block.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.kzo_decode_block.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.kzo_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_size_t,
                                   C.POINTER(C.c_size_t), C.POINTER(C.c_double)]
        L.kzo_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_double)]
        L.kzo_parse_transform.argtypes = [C.c_char_p]
        L.kzo_parse_transform.restype = C.c_uint64
        L.kzo_parse_entropy.argtypes = [C.c_char_p]
        L.kzo_xxhash32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
        L.kzo_xxhash32.restype = C.c_uint32
        L.kzo_xxhash64.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64]
        L.kzo_xxhash64.restype = C.c_uint64
        L.kzo_varint_len.argtypes = [C.c_uint32]
        L.kzo_normalize.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.kzo_entropy1024.argtypes = [C.c_void_p, C.c_size_t]
        _lib = L
    return _lib


class OracleError(RuntimeError):
    def __init__(self, rc):
        self.code = -rc
        super().__init__("oracle error %d: %s" % (-rc, lib().kzo_last_error().decode()))


def _arr(b):
    a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, dtype=np.uint8)
    return a


def _ptr(a):
    return a.ctypes.data if a.size else None


def entropy_encode(etype, data):
    """-> (bytes, nbits)"""
    a = _arr(data)
    cap = a.size + a.size // 4 + 70000 + 110000 * (a.size // (4 << 20) + 1)
    out = np.empty(cap, np.uint8)
    bits = C.c_uint64(0)
    rc = lib().kzo_entropy_encode(etype, _ptr(a), a.size, out.ctypes.data, cap, C.byref(bits))
    if rc:
        raise OracleError(rc)
    return out[: (bits.value + 7) // 8].copy(), bits.value


def entropy_decode(etype, stream, n):
    """-> (decoded bytes array, consumed bits)"""
    s = _arr(stream)
    out = np.empty(max(n, 1), np.uint8)
    used = C.c_uint64(0)
    rc = lib().kzo_entropy_decode(etype, _ptr(s), s.size, out.ctypes.data, n, C.byref(used))
    if rc:
        raise OracleError(rc)
    return out[:n], used.value


def transform_forward(ttype, data, data_type=0, block_size=0):
    """-> (out bytes or None when the transform asks to be skipped, data_type after). block_size = the stream's block size
    (ctx["blockSize"], only read by TEXT); 0 = len(data)."""
    a = _arr(data)
    lib().kzo_set_stream_block_size(block_size)
    cap = max(lib().kzo_transform_max_encoded_len(ttype, a.size), a.size) + 64
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    dt = C.c_int(data_type)
    rc = lib().kzo_transform_forward(ttype, data_type, _ptr(a), a.size, out.ctypes.data, cap, C.byref(n), C.byref(dt))
    if rc < 0:
        raise OracleError(rc)
    if rc == 1:
        return None, dt.value
    return out[: n.value].copy(), dt.value


def transform_inverse(ttype, data, cap, data_type=0, block_size=0):
    a = _arr(data)
    lib().kzo_set_stream_block_size(block_size)
    out = np.empty(max(cap, 1), np.uint8)
    n = C.c_size_t(0)
    rc = lib().kzo_transform_inverse(ttype, data_type, _ptr(a), a.size, out.ctypes.data, cap, C.byref(n))
    if rc:
        raise OracleError(rc)
    return out[: n.value].copy()


def bwt_forward_raw(data):
    a = _arr(data)
    out = np.empty(max(a.size, 1), np.uint8)
    prim = np.zeros(8, np.uint32)
    lib().kzo_bwt_forward_raw(_ptr(a), out.ctypes.data, a.size, prim.ctypes.data)
    return out[: a.size], prim


def bwt_inverse_raw(data, prim):
    a = _arr(data)
    out = np.empty(max(a.size, 1), np.uint8)
    p = np.ascontiguousarray(prim, dtype=np.uint32)
    rc = lib().kzo_bwt_inverse_raw(_ptr(a), out.ctypes.data, a.size, p.ctypes.data)
    if rc:
        raise OracleError(-13)
    return out[: a.size]


def encode_block(data, transform48, entropy, checksum_bits=0, skip_blocks=False):
    a = _arr(data)
    cap = a.size + a.size // 4 + 70000 + 110000 * (a.size // (4 << 20) + 1)
    out = np.empty(cap, np.uint8)
    bits = C.c_uint64(0)
    rc = lib().kzo_encode_block(_ptr(a), a.size, transform48, entropy, checksum_bits, int(skip_blocks), out.ctypes.data, cap, C.byref(bits))
    if rc:
        raise OracleError(rc)
    return out[: (bits.value + 7) // 8].copy(), bits.value


def decode_block(payload, bits, transform48, entropy, checksum_bits, block_size):
    s = _arr(payload)
    cap = block_size + block_size // 2 + 4096
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    rc = lib().kzo_decode_block(_ptr(s), bits, transform48, entropy, checksum_bits, block_size, out.ctypes.data, cap, C.byref(n))
    if rc:
        raise OracleError(rc)
    return out[: n.value].copy()


def compress(data, transform="NONE", entropy="NONE", block_size=4 << 20, checksum_bits=0, jobs=1, input_size=0, timing=None):
    a = _arr(data)
    t48 = parse_transform(transform) if isinstance(transform, str) else transform
    et = parse_entropy(entropy) if isinstance(entropy, str) else entropy
    cap = a.size + a.size // 4 + 70000 + (64 + 110000) * (a.size // max(block_size, 1) + 1)
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    secs = C.c_double(0)
    rc = lib().kzo_compress(_ptr(a), a.size, t48, et, block_size, checksum_bits, jobs, input_size, out.ctypes.data, cap, C.byref(n), C.byref(secs))
    if rc:
        raise OracleError(rc)
    if timing is not None:
        timing.append(secs.value)
    return out[: n.value].copy()


def decompress(stream, out_cap, jobs=1, timing=None):
    s = _arr(stream)
    out = np.empty(max(out_cap, 1), np.uint8)
    n = C.c_size_t(0)
    secs = C.c_double(0)
    rc = lib().kzo_decompress(_ptr(s), s.size, jobs, out.ctypes.data, out_cap, C.byref(n), C.byref(secs))
    if rc:
        raise OracleError(rc)
    if timing is not None:
        timing.append(secs.value)
    return out[: n.value]


def parse_transform(names):
    v = lib().kzo_parse_transform(names.encode())
    if v == 0xFFFFFFFFFFFFFFFF:
        raise ValueError("Unknown transform type: %r" % names)
    return v


def parse_entropy(name):
    v = lib().kzo_parse_entropy(name.encode())
    if v < 0:
        raise ValueError("Unsupported entropy codec type: %r" % name)
    return v


def xxhash32(data, seed=0):
    a = _arr(data)
    return lib().kzo_xxhash32(_ptr(a), a.size, seed)


def xxhash64(data, seed=0):
    a = _arr(data)
    return lib().kzo_xxhash64(_ptr(a), a.size, seed)
