"""ctypes bindings for the CPU checkers under oracle/ (TEST INFRASTRUCTURE).

`load("port")`  -> oracle/liboracle.so       (plain-C restatement)
`load("ref")`   -> oracle/_ref/libsela_ref.so (unmodified reference, if built)

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this.
"""
import ctypes as C
import hashlib
import pathlib
import subprocess

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
FRAME = 2048


class Desc(C.Structure):
    _fields_ = [
        ("channel", C.c_uint8), ("subframe_type", C.c_uint8), ("parent_channel", C.c_uint8),
        ("refl_rice_param", C.c_uint8), ("refl_words", C.c_uint16), ("lpc_order", C.c_uint8),
        ("res_rice_param", C.c_uint8), ("res_words", C.c_uint16), ("samples", C.c_uint16),
        ("reserved", C.c_uint32), ("refl_offset", C.c_uint64), ("res_offset", C.c_uint64),
    ]


DESC_DTYPE = np.dtype([
    ("channel", "u1"), ("subframe_type", "u1"), ("parent_channel", "u1"),
    ("refl_rice_param", "u1"), ("refl_words", "<u2"), ("lpc_order", "u1"),
    ("res_rice_param", "u1"), ("res_words", "<u2"), ("samples", "<u2"),
    ("reserved", "<u4"), ("refl_offset", "<u8"), ("res_offset", "<u8"),
], align=True)
assert DESC_DTYPE.itemsize == C.sizeof(Desc) == 32, (DESC_DTYPE.itemsize, C.sizeof(Desc))


def build(force=False):
    """make -C oracle (liboracle.so always; _ref only where the reference sources are present)."""
    if force or not (ORACLE_DIR / "liboracle.so").exists():
        subprocess.run(["make", "-C", str(ORACLE_DIR)], check=True, capture_output=True)


def have_ref():
    return (ORACLE_DIR / "_ref" / "libsela_ref.so").exists()


_p = lambda a, t: a.ctypes.data_as(C.POINTER(t))


class Oracle:
    def __init__(self, path):
        self.lib = L = C.CDLL(str(path))
        L.sela_oracle_kind.restype = C.c_char_p
        L.sela_oracle_rice_encode.restype = C.c_size_t
        L.sela_oracle_rice_size.restype = C.c_size_t
        L.sela_oracle_time_encode.restype = C.c_double
        L.sela_oracle_time_decode.restype = C.c_double
        L.sela_oracle_rice_encode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t]
        L.sela_oracle_rice_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p]
        L.sela_oracle_lpc_analyse.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 6
        L.sela_oracle_lpc_synthesise.argtypes = [C.c_void_p, C.c_size_t, C.c_uint8, C.c_void_p, C.c_void_p]
        L.sela_oracle_lpc_coefficients.argtypes = [C.c_void_p, C.c_uint8, C.c_void_p]
        L.sela_oracle_encode_frames.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                C.c_size_t, C.c_void_p, C.c_int]
        L.sela_oracle_decode_frames.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int]
        L.sela_oracle_time_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.sela_oracle_time_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]
        L.sela_oracle_frame_encode_i32.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                   C.c_size_t, C.c_void_p]
        L.sela_oracle_frame_decode_i32.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        self.kind = L.sela_oracle_kind().decode()
        self.cores = L.sela_oracle_online_cores()

    # ---- stage level ------------------------------------------------------
    def lpc_analyse(self, s, want_internals=False):
        s = np.ascontiguousarray(s, dtype=np.int32)
        n = s.size
        order = C.c_uint8(0)
        q = np.zeros(100, np.int32)
        c = np.zeros(101, np.int64)
        res = np.zeros(n, np.int32)
        refl = np.zeros(100, np.float64)
        ac = np.zeros(101, np.float64)
        self.lib.sela_oracle_lpc_analyse(s.ctypes.data, n, C.addressof(order), q.ctypes.data, c.ctypes.data,
                                         res.ctypes.data, refl.ctypes.data, ac.ctypes.data)
        o = order.value
        out = dict(order=o, q=q[:o].copy(), c=c[:o + 1].copy(), res=res)
        if want_internals:
            out.update(refl=refl, ac=ac)
        return out

    def lpc_coefficients(self, q, order):
        q = np.ascontiguousarray(q, dtype=np.int32)
        c = np.zeros(order + 1, np.int64)
        self.lib.sela_oracle_lpc_coefficients(q.ctypes.data, order, c.ctypes.data)
        return c

    def lpc_synthesise(self, res, order, q):
        res = np.ascontiguousarray(res, dtype=np.int32)
        q = np.ascontiguousarray(q, dtype=np.int32)
        s = np.zeros(res.size, np.int32)
        self.lib.sela_oracle_lpc_synthesise(res.ctypes.data, res.size, order, q.ctypes.data, s.ctypes.data)
        return s

    def rice_encode(self, x):
        x = np.ascontiguousarray(x, dtype=np.int32)
        k = C.c_uint32(0)
        cap = 1 << 16
        while True:
            words = np.zeros(cap, np.uint32)
            n = self.lib.sela_oracle_rice_encode(x.ctypes.data, x.size, C.addressof(k), words.ctypes.data, cap)
            if n <= cap:
                return k.value, words[:n].copy()
            cap = n

    def rice_decode(self, words, k, count):
        words = np.ascontiguousarray(words, dtype=np.uint32)
        padded = np.concatenate([words, np.zeros(4, np.uint32)])
        out = np.zeros(count, np.int32)
        self.lib.sela_oracle_rice_decode(padded.ctypes.data, words.size, k, count, out.ctypes.data)
        return out

    # ---- frame / batch level ---------------------------------------------
    def encode_frames(self, pcm, channels, threads=0):
        """pcm: int16 array of n_frames*2048*channels interleaved samples."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16).reshape(-1)
        n_frames = pcm.size // (FRAME * channels)
        assert n_frames * FRAME * channels == pcm.size
        descs = np.zeros(n_frames * channels, DESC_DTYPE)
        cap = n_frames * channels * 2200 + 4096
        while True:
            words = np.zeros(cap, np.uint32)
            used = C.c_size_t(0)
            rc = self.lib.sela_oracle_encode_frames(pcm.ctypes.data, n_frames, channels, descs.ctypes.data,
                                                    words.ctypes.data, cap, C.addressof(used), threads)
            if rc == 0:
                return descs, words[:used.value].copy()
            cap *= 4

    def decode_frames(self, descs, words, channels, threads=0):
        descs = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
        words = np.concatenate([np.ascontiguousarray(words, dtype=np.uint32), np.zeros(4, np.uint32)])
        n_frames = descs.size // channels
        pcm = np.zeros(n_frames * FRAME * channels, np.int16)
        self.lib.sela_oracle_decode_frames(descs.ctypes.data, n_frames, channels, words.ctypes.data,
                                           pcm.ctypes.data, threads)
        return pcm

    def frame_encode_i32(self, planes):
        planes = [np.ascontiguousarray(p, dtype=np.int32) for p in planes]
        ch, n = len(planes), planes[0].size
        ptrs = (C.c_void_p * ch)(*[p.ctypes.data for p in planes])
        descs = np.zeros(ch, DESC_DTYPE)
        cap = 1 << 18
        while True:
            words = np.zeros(cap, np.uint32)
            used = C.c_size_t(0)
            rc = self.lib.sela_oracle_frame_encode_i32(ptrs, ch, n, descs.ctypes.data, words.ctypes.data, cap,
                                                       C.addressof(used))
            if rc == 0:
                return descs, words[:used.value].copy()
            cap *= 4

    def frame_decode_i32(self, descs, words):
        descs = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
        words = np.concatenate([np.ascontiguousarray(words, dtype=np.uint32), np.zeros(4, np.uint32)])
        ch = descs.size
        n = int(descs["samples"].max())
        planes = [np.zeros(max(n, 1), np.int32) for _ in range(ch)]
        ptrs = (C.c_void_p * ch)(*[p.ctypes.data for p in planes])
        self.lib.sela_oracle_frame_decode_i32(descs.ctypes.data, ch, words.ctypes.data, ptrs)
        return planes

    def time_encode(self, pcm, channels, threads=0):
        pcm = np.ascontiguousarray(pcm, dtype=np.int16).reshape(-1)
        return self.lib.sela_oracle_time_encode(pcm.ctypes.data, pcm.size // (FRAME * channels), channels, threads)

    def time_decode(self, descs, words, channels, threads=0):
        descs = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
        words = np.concatenate([np.ascontiguousarray(words, dtype=np.uint32), np.zeros(4, np.uint32)])
        return self.lib.sela_oracle_time_decode(descs.ctypes.data, descs.size // channels, channels,
                                                words.ctypes.data, threads)


_cache = {}


def load(which="port"):
    build()
    if which not in _cache:
        path = ORACLE_DIR / ("liboracle.so" if which == "port" else "_ref/libsela_ref.so")
        _cache[which] = Oracle(path)
    return _cache[which]


def best():
    """The strongest checker available: the compiled reference if present, else the port."""
    return load("ref") if have_ref() else load("port")


def golden(name):
    """tests/golden/<name>.npz, loaded once."""
    if name not in _golden:
        _golden[name] = np.load(ROOT / "tests" / "golden" / (name + ".npz"))
    return _golden[name]


_golden = {}


def digest(a):
    """Short SHA-256 of an array's dtype and bytes: how tests/golden stores reference outputs too large to keep."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.dtype.str.encode() + a.tobytes()).hexdigest()[:32]


def fnv1a32(words):
    """FNV-1a-32 over the little-endian bytes (the hash SURVEY.md 8a's KAT table uses)."""
    h = 0x811C9DC5
    for b in np.ascontiguousarray(words, dtype="<u4").tobytes():
        h = ((h ^ b) * 0x01000193) & 0xFFFFFFFF
    return h
