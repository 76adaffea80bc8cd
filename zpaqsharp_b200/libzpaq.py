"""ctypes binding of libzpaqb200.so plus a thin mirror of the reference's LibZPAQ surface.

The product is the shared library (CUDA kernels + host scheduler behind the C ABI declared in
include/zpaqb200.h).  This module is the Python-side equivalent of the C# P/Invoke facade in
bindings/csharp/: the same names and argument meaning as LibZPAQ.cs (Compress :84,
compressBlock :117, decompress :65) and Compressor.startBlock(int) (Compressor.cs:45), with
errors raised as exceptions the way LibZPAQ.error() does (LibZPAQ.cs:22-24).

Nothing here computes on the CPU: every call that touches block data goes to the GPU through the
C ABI, and loading fails loudly when the library has not been built.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzpaqb200.so")

E_ARG, E_CONFIG, E_CUDA, E_NOMEM, E_OUTPUT, E_CORRUPT, E_UNSUPPORTED = -1, -2, -3, -4, -5, -6, -7

# Every symbol include/zpaqb200.h declares (tests check that the library exports all of them).
ABI_SYMBOLS = [
    "zpq_create", "zpq_destroy", "zpq_last_error", "zpq_set_stream", "zpq_set_max_resident",
    "zpq_make_config", "zpq_expand_method", "zpq_compile_config", "zpq_builtin_model", "zpq_block_memory",
    "zpq_device_state_bytes", "zpq_device_state_bytes_for", "zpq_compress_blocks", "zpq_compress_blocks_level", "zpq_compress_blocks_model",
    "zpq_compress_blocks_model_dev", "zpq_find_blocks", "zpq_decompress_blocks", "zpq_decompressed_bound",
    "zpq_get_stats", "zpq_version", "zpq_specialize_model", "zpq_encoder_plan", "zpq_post_kind", "zpq_specialize_pcomp",
    "zpq_scrypt", "zpq_stretch_key", "zpq_aes_ctr", "zpq_aes_ctr_dev",
]


class ZpaqError(RuntimeError):
    """LibZPAQ.error(msg) (LibZPAQ.cs:22-24): the library reports, the host throws."""

    def __init__(self, code: int, msg: str):
        super().__init__("%s (code %d)" % (msg, code))
        self.code = code


class Stats(C.Structure):
    _fields_ = [("h2d_ms", C.c_double), ("kernel_ms", C.c_double), ("d2h_ms", C.c_double), ("total_ms", C.c_double),
                ("codec_kernel_ms", C.c_double), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("launches", C.c_uint32), ("resident_blocks", C.c_uint32), ("state_bytes_per_block", C.c_uint64),
                ("kernel", C.c_char * 96), ("post_kernel_ms", C.c_double),
                ("post_native_blocks", C.c_uint32), ("post_interpreted_blocks", C.c_uint32),
                ("post_compiled_blocks", C.c_uint32), ("reserved0", C.c_uint32)]


_lib = None


def load():
    """Load libzpaqb200.so (built by zpaqsharp_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ZpaqError(E_CUDA, "libzpaqb200.so is not built; run `python -m zpaqsharp_b200.build` "
                                "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    u8p, u64p, i32p = C.c_void_p, C.c_void_p, C.POINTER(C.c_int)
    L.zpq_version.restype = C.c_char_p
    L.zpq_last_error.restype = C.c_char_p
    L.zpq_last_error.argtypes = [C.c_void_p]
    L.zpq_create.argtypes = [i32p, C.c_int, C.POINTER(C.c_void_p)]
    L.zpq_destroy.argtypes = [C.c_void_p]
    L.zpq_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.zpq_set_max_resident.argtypes = [C.c_void_p, C.c_uint32]
    L.zpq_make_config.restype = C.c_int64
    L.zpq_make_config.argtypes = [C.c_char_p, i32p, C.c_char_p, C.c_uint64]
    L.zpq_expand_method.restype = C.c_int64
    L.zpq_expand_method.argtypes = [C.c_char_p, u8p, C.c_uint64, C.c_char_p, C.c_uint64]
    L.zpq_compile_config.argtypes = [C.c_char_p, i32p, u8p, C.c_uint64, C.POINTER(C.c_uint64), u8p, C.c_uint64,
                                     C.POINTER(C.c_uint64)]
    L.zpq_builtin_model.restype = C.c_int64
    L.zpq_builtin_model.argtypes = [C.c_int, u8p, C.c_uint64]
    L.zpq_block_memory.restype = C.c_double
    L.zpq_block_memory.argtypes = [u8p, C.c_uint64]
    L.zpq_device_state_bytes.restype = C.c_int64
    L.zpq_device_state_bytes.argtypes = [u8p, C.c_uint64, C.c_int]
    L.zpq_compress_blocks.argtypes = [C.c_void_p, u8p, u64p, C.c_uint32, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int,
                                      u8p, C.c_uint64, u64p]
    L.zpq_compress_blocks_level.argtypes = [C.c_void_p, C.c_int, u8p, u64p, C.c_uint32, C.c_char_p, C.c_char_p,
                                            C.c_int, C.c_int, u8p, C.c_uint64, u64p]
    L.zpq_compress_blocks_model.argtypes = [C.c_void_p, u8p, C.c_uint64, u8p, C.c_uint64, i32p, u8p, u64p, C.c_uint32,
                                            C.c_char_p, C.c_char_p, C.c_int, C.c_int, u8p, C.c_uint64, u64p]
    L.zpq_compress_blocks_model_dev.argtypes = [C.c_void_p, u8p, C.c_uint64, u8p, C.c_uint64, i32p, u8p, u64p,
                                                C.c_uint32, C.c_int, C.c_int, u8p, C.c_uint64, u64p]
    L.zpq_find_blocks.restype = C.c_int64
    L.zpq_find_blocks.argtypes = [u8p, C.c_uint64, u64p, C.c_uint64]
    L.zpq_decompress_blocks.argtypes = [C.c_void_p, u8p, u64p, C.c_uint32, u8p, C.c_uint64, u64p, u8p, u8p]
    L.zpq_decompressed_bound.restype = C.c_int64
    L.zpq_decompressed_bound.argtypes = [u8p, u64p, C.c_uint32]
    L.zpq_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.zpq_specialize_model.restype = C.c_int64
    L.zpq_specialize_model.argtypes = [u8p, C.c_uint64, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64]
    L.zpq_scrypt.argtypes = [u8p, C.c_uint64, u8p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, u8p, C.c_uint64]
    L.zpq_stretch_key.argtypes = [u8p, u8p, u8p]
    L.zpq_aes_ctr.argtypes = [C.c_void_p, u8p, C.c_int, u8p, u8p, C.c_uint64, C.c_uint64]
    L.zpq_aes_ctr_dev.argtypes = [C.c_void_p, u8p, C.c_int, u8p, u8p, C.c_uint64, C.c_uint64]
    _lib = L
    return L


def _buf(data):
    """bytes / bytearray / numpy uint8 array -> (address, length, keepalive)."""
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data, dtype=np.uint8)
        return a.ctypes.data, a.size, a
    a = np.frombuffer(data, dtype=np.uint8)
    return a.ctypes.data, a.size, a


def _raise(ctx, code):
    msg = load().zpq_last_error(ctx) or b""
    raise ZpaqError(code, msg.decode(errors="replace"))


# ---- host front end (no device needed) --------------------------------------------------------
def make_config(method: str):
    """LibZPAQ.makeConfig, LibZPAQ.cs:388 -> (config text, args[9])."""
    L = load()
    args = (C.c_int * 9)()
    n = L.zpq_make_config(method.encode(), args, None, 0)
    if n < 0:
        _raise(None, n)
    buf = C.create_string_buffer(n + 1)
    L.zpq_make_config(method.encode(), args, buf, n + 1)
    return buf.value.decode(), list(args)


def expand_method(method: str, block: bytes) -> str:
    """Level-digit expansion inside compressBlock, LibZPAQ.cs:128-283."""
    L = load()
    p, n, keep = _buf(block)
    buf = C.create_string_buffer(4096)
    r = L.zpq_expand_method(method.encode(), p, n, buf, 4096)
    if r < 0:
        _raise(None, r)
    return buf.value.decode()


def compile_config(text: str, args=None):
    """Compiler(config, args, hz, pz), Compiler.cs:13 -> (header bytes, pcomp bytes)."""
    L = load()
    a = (C.c_int * 9)(*(args or [0] * 9))
    hdr = C.create_string_buffer(70000)
    pc = C.create_string_buffer(70000)
    hl, pl = C.c_uint64(0), C.c_uint64(0)
    r = L.zpq_compile_config(text.encode(), a, hdr, 70000, C.byref(hl), pc, 70000, C.byref(pl))
    if r < 0:
        _raise(None, r)
    return hdr.raw[:hl.value], pc.raw[:pl.value]


def builtin_model(level: int) -> bytes:
    """Model bytes of Compressor.startBlock(int level), Compressor.cs:45-83."""
    L = load()
    buf = C.create_string_buffer(1024)
    n = L.zpq_builtin_model(level, buf, 1024)
    if n < 0:
        _raise(None, n)
    return buf.raw[:n]


def block_memory(hdr: bytes) -> float:
    """ZPAQL.memory(), ZPAQL.cs:58-81."""
    return load().zpq_block_memory(hdr, len(hdr))


def device_state_bytes(hdr: bytes, for_decode: bool = False, max_block_bytes: int = 0) -> int:
    """Device state of one resident block; with max_block_bytes, as the scheduler sizes it for a batch of such blocks."""
    L = load()
    if max_block_bytes:
        L.zpq_device_state_bytes_for.restype = C.c_int64
        L.zpq_device_state_bytes_for.argtypes = [C.c_char_p, C.c_uint64, C.c_int, C.c_uint64]
        return L.zpq_device_state_bytes_for(hdr, len(hdr), 1 if for_decode else 0, max_block_bytes)
    return L.zpq_device_state_bytes(hdr, len(hdr), 1 if for_decode else 0)


def encoder_plan(hdr: bytes, smem_bytes: int = 232448, blocks_per_sm: int = 32) -> dict:
    """How the role-split encoder would run this model (host only): see zpq_encoder_plan in include/zpaqb200.h."""
    out = (C.c_int32 * 8)()
    L = load()
    L.zpq_encoder_plan.argtypes = [C.c_char_p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32)]
    L.zpq_encoder_plan.restype = C.c_int
    rc = L.zpq_encoder_plan(hdr, len(hdr), smem_bytes, blocks_per_sm, out)
    if rc:
        raise ZpaqError(rc, "zpq_encoder_plan failed")
    keys = ["applies", "lanes_per_block", "roles", "blocks_per_sm", "smem_per_block", "coder_delay", "mixer_role", "warps_per_cta"]
    return dict(zip(keys, [int(v) for v in out]))


def post_kind(ph: int, pm: int, pcomp: bytes) -> int:
    """How the decoder restores a block with this PCOMP program: 0 = interpreted, else kind | e8 << 4 | param << 8 (see the header)."""
    L = load()
    L.zpq_post_kind.restype = C.c_int64
    L.zpq_post_kind.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint64]
    return int(L.zpq_post_kind(ph, pm, bytes(pcomp), len(pcomp)))


def specialize_pcomp(ph: int, pm: int, pcomp: bytes):
    """Translate + NVRTC-compile a PCOMP program -> (cubin size or error, source, log); needs no GPU."""
    L = load()
    L.zpq_specialize_pcomp.restype = C.c_int64
    L.zpq_specialize_pcomp.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64]
    src = C.create_string_buffer(1 << 20)
    log = C.create_string_buffer(1 << 16)
    n = L.zpq_specialize_pcomp(ph, pm, bytes(pcomp), len(pcomp), src, 1 << 20, log, 1 << 16)
    return n, src.value.decode(), log.value.decode(errors="replace")


def specialize_model(hdr: bytes):
    """Generate + NVRTC-compile the specialised kernels of a header -> (cubin size or error, source, log)."""
    L = load()
    src = C.create_string_buffer(1 << 20)
    log = C.create_string_buffer(1 << 16)
    n = L.zpq_specialize_model(hdr, len(hdr), src, 1 << 20, log, 1 << 16)
    return n, src.value.decode(), log.value.decode(errors="replace")


def find_blocks(archive) -> list:
    """Decompresser.findBlock over a whole archive, Decompresser.cs:29-58 -> [(start, end), ...]."""
    L = load()
    p, n, keep = _buf(archive)
    cnt = L.zpq_find_blocks(p, n, None, 0)
    if cnt < 0:
        _raise(None, cnt)
    offs = np.zeros(2 * max(cnt, 1), dtype=np.uint64)
    L.zpq_find_blocks(p, n, offs.ctypes.data, cnt)
    return [(int(offs[2 * i]), int(offs[2 * i + 1])) for i in range(cnt)]


# ---- key derivation (host, no device needed) ------------------------------------------------------
def scrypt(pw: bytes, salt: bytes, n: int, r: int, p: int, dklen: int) -> bytes:
    """libzpaq scrypt (RFC 7914), which stretchKey calls (StretchKey.cs:13-163)."""
    out = C.create_string_buffer(max(dklen, 1))
    rc = load().zpq_scrypt(bytes(pw), len(pw), bytes(salt), len(salt), n, r, p, out, dklen)
    if rc != 0:
        _raise(None, rc)
    return out.raw[:dklen]


def stretch_key(in32: bytes, salt32: bytes) -> bytes:
    """libzpaq stretchKey (StretchKey.cs:13-163): scrypt(in32, salt32, 16384, 8, 1, 32); in32 is SHA-256 of the password."""
    if len(in32) != 32 or len(salt32) != 32:
        raise ZpaqError(E_ARG, "stretch_key takes 32-byte key and salt")
    out = C.create_string_buffer(32)
    rc = load().zpq_stretch_key(bytes(in32), bytes(salt32), out)
    if rc != 0:
        _raise(None, rc)
    return out.raw


def _aes_key_iv(key, iv):
    key = bytes(key)
    if iv is not None and len(iv) != 8:
        raise ZpaqError(E_ARG, "the AES-CTR iv is 8 bytes")
    return key, (bytes(iv) if iv is not None else None)


def block_size_of(method: str) -> int:
    """Block size LibZPAQ.Compress derives from the method string, LibZPAQ.cs:87-94."""
    bs = 4
    if len(method) > 1 and method[1].isdigit():
        bs = int(method[1])
        if len(method) > 2 and method[2].isdigit():
            bs = bs * 10 + int(method[2])
        bs = min(bs, 11)
    return (0x100000 << bs) - 4096


def split_offsets(n: int, block_size: int) -> np.ndarray:
    offs = list(range(0, n, block_size)) + [n]
    if n == 0:
        offs = [0]
    return np.asarray(offs, dtype=np.uint64)


# ---- device context ---------------------------------------------------------------------------
class Context:
    """One zpq_ctx: owns device memory, streams and tables on the chosen GPU(s)."""

    def __init__(self, devices=None):
        L = load()
        self._h = C.c_void_p()
        if devices is None:
            rc = L.zpq_create(None, 0, C.byref(self._h))
        else:
            ids = (C.c_int * len(devices))(*devices)
            rc = L.zpq_create(ids, len(devices), C.byref(self._h))
        if rc != 0:
            self._h = None
            _raise(None, rc)

    def close(self):
        if getattr(self, "_h", None):
            try:
                load().zpq_destroy(self._h)
            except TypeError:              # interpreter shutdown: the module globals are gone, the process frees the device
                pass
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream: int | None):
        load().zpq_set_stream(self._h, C.c_void_p(cuda_stream or 0))

    def set_max_resident(self, n: int):
        load().zpq_set_max_resident(self._h, n)

    def stats(self) -> Stats:
        s = Stats()
        load().zpq_get_stats(self._h, C.byref(s))
        return s

    # -- compression --
    def _out(self, total_in: int, nb: int, out):
        cap = total_in + total_in // 4 + 8192 * (nb + 1) + 65536
        if out is None:
            out = np.empty(cap, dtype=np.uint8)
        return out, out.size

    def compress_blocks(self, data, offsets, method: str, filename=None, comment=None, dosha1=True, out=None):
        """LibZPAQ.compressBlock for every block, LibZPAQ.cs:117.  Returns (archive bytes view, out offsets)."""
        L = load()
        p, n, keep = _buf(data)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        nb = offs.size - 1
        out, cap = self._out(int(offs[-1] - offs[0]), nb, out)
        ooff = np.zeros(nb + 1, dtype=np.uint64)
        rc = L.zpq_compress_blocks(self._h, p, offs.ctypes.data, nb, method.encode(),
                                   filename.encode() if filename else None, comment.encode() if comment else None,
                                   1 if dosha1 else 0, out.ctypes.data, cap, ooff.ctypes.data)
        if rc != 0:
            _raise(self._h, rc)
        return out[:int(ooff[nb])], ooff

    def compress_blocks_level(self, data, offsets, level: int, filename=None, comment=None, dosha1=True,
                              with_tag=True, out=None):
        """Compressor.startBlock(level) .. endBlock for every block, Compressor.cs:45-299."""
        L = load()
        p, n, keep = _buf(data)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        nb = offs.size - 1
        out, cap = self._out(int(offs[-1] - offs[0]), nb, out)
        ooff = np.zeros(nb + 1, dtype=np.uint64)
        rc = L.zpq_compress_blocks_level(self._h, level, p, offs.ctypes.data, nb,
                                         filename.encode() if filename else None,
                                         comment.encode() if comment else None, 1 if dosha1 else 0,
                                         1 if with_tag else 0, out.ctypes.data, cap, ooff.ctypes.data)
        if rc != 0:
            _raise(self._h, rc)
        return out[:int(ooff[nb])], ooff

    def compress_blocks_model(self, data, offsets, hdr: bytes, pcomp: bytes = b"", args=None, filename=None,
                              comment=None, dosha1=True, with_tag=True, out=None):
        """Compressor.startBlock(hcomp bytes) path, Compressor.cs:85-99."""
        L = load()
        p, n, keep = _buf(data)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        nb = offs.size - 1
        out, cap = self._out(int(offs[-1] - offs[0]) + len(pcomp) * nb, nb, out)
        ooff = np.zeros(nb + 1, dtype=np.uint64)
        a = (C.c_int * 9)(*(args or [0] * 9))
        rc = L.zpq_compress_blocks_model(self._h, hdr, len(hdr), pcomp if pcomp else None, len(pcomp), a, p,
                                         offs.ctypes.data, nb, filename.encode() if filename else None,
                                         comment.encode() if comment else None, 1 if dosha1 else 0,
                                         1 if with_tag else 0, out.ctypes.data, cap, ooff.ctypes.data)
        if rc != 0:
            _raise(self._h, rc)
        return out[:int(ooff[nb])], ooff

    def compress_blocks_model_dev(self, d_in_ptr: int, offsets, hdr: bytes, d_out_ptr: int, out_cap: int,
                                  pcomp: bytes = b"", args=None, dosha1=True, with_tag=True):
        """Device-resident variant: d_in_ptr / d_out_ptr are CUDA device addresses."""
        L = load()
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        nb = offs.size - 1
        ooff = np.zeros(nb + 1, dtype=np.uint64)
        a = (C.c_int * 9)(*(args or [0] * 9))
        rc = L.zpq_compress_blocks_model_dev(self._h, hdr, len(hdr), pcomp if pcomp else None, len(pcomp), a,
                                             C.c_void_p(d_in_ptr), offs.ctypes.data, nb, 1 if dosha1 else 0,
                                             1 if with_tag else 0, C.c_void_p(d_out_ptr), out_cap, ooff.ctypes.data)
        if rc != 0:
            _raise(self._h, rc)
        return ooff

    # -- encryption (libzpaq AES_CTR) --
    def aes_ctr(self, buf, key: bytes, iv: bytes | None = None, offset: int = 0):
        """AES_CTR(key, iv).encrypt(buf, len(buf), offset) on the GPU, in place on a writable buffer (bytearray, numpy uint8,
        ...); returns buf.  Encrypting and decrypting are the same call."""
        a = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
        if a.dtype != np.uint8 or not a.flags.c_contiguous or not a.flags.writeable:
            raise TypeError("aes_ctr works in place: pass a writable, contiguous uint8 buffer")
        key, iv = _aes_key_iv(key, iv)
        rc = load().zpq_aes_ctr(self._h, key, len(key), iv, a.ctypes.data if a.size else None, a.size, offset)
        if rc != 0:
            _raise(self._h, rc)
        return buf

    def aes_ctr_dev(self, d_ptr: int, n: int, key: bytes, iv: bytes | None = None, offset: int = 0):
        """The same on n bytes at CUDA device address d_ptr (device 0 of the context), on the context's stream."""
        key, iv = _aes_key_iv(key, iv)
        rc = load().zpq_aes_ctr_dev(self._h, key, len(key), iv, C.c_void_p(d_ptr or None), n, offset)
        if rc != 0:
            _raise(self._h, rc)

    # -- decompression --
    def decompress_blocks(self, archive, offsets, out=None):
        """LibZPAQ.decompress for the given blocks, LibZPAQ.cs:65.  Returns (bytes view, out offsets,
        sha1 status per block, block status per block)."""
        L = load()
        p, n, keep = _buf(archive)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        nb = offs.size - 1
        if out is None:
            bound = L.zpq_decompressed_bound(p, offs.ctypes.data, nb)
            if bound < 0:
                _raise(None, bound)
            out = np.empty(max(int(bound), 16), dtype=np.uint8)
        ooff = np.zeros(nb + 1, dtype=np.uint64)
        sha = np.zeros(max(nb, 1), dtype=np.uint8)
        bst = np.zeros(max(nb, 1), dtype=np.uint8)
        rc = L.zpq_decompress_blocks(self._h, p, offs.ctypes.data, nb, out.ctypes.data, out.size, ooff.ctypes.data,
                                     sha.ctypes.data, bst.ctypes.data)
        if rc != 0:
            err = ZpaqError(rc, (L.zpq_last_error(self._h) or b"").decode(errors="replace"))
            err.block_status = bst[:nb].copy()
            raise err
        return out[:int(ooff[nb])], ooff, sha[:nb], bst[:nb]


# ---- LibZPAQ-style one-call API -----------------------------------------------------------------
_default_ctx = None


def _ctx() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


def compressBlock(data: bytes, method: str, filename=None, comment=None, dosha1=True) -> bytes:
    """LibZPAQ.compressBlock, LibZPAQ.cs:117: one block, whatever its size."""
    out, _ = _ctx().compress_blocks(data, np.asarray([0, len(data)], dtype=np.uint64), method, filename, comment,
                                    dosha1)
    return out.tobytes()


def compress(data: bytes, method: str = "14,128,0", filename=None, comment=None, dosha1=True) -> bytes:
    """LibZPAQ.Compress, LibZPAQ.cs:84: split by the method's block size, code every block."""
    offs = split_offsets(len(data), block_size_of(method))
    if offs.size < 2:
        return b""
    out, _ = _ctx().compress_blocks(data, offs, method, filename, comment, dosha1)
    return out.tobytes()


def decompress(archive: bytes) -> bytes:
    """LibZPAQ.decompress, LibZPAQ.cs:65: every block and segment of the archive, in order."""
    blocks = find_blocks(archive)
    if not blocks:
        return b""
    # decode each block from its "zPQ"; the bytes between blocks (tags) are not data
    out = bytearray()
    offs = np.asarray([b[0] for b in blocks] + [blocks[-1][1]], dtype=np.uint64)
    # blocks are contiguous up to their tags; give each block exactly its own range
    ranges = np.zeros(len(blocks) + 1, dtype=np.uint64)
    a = np.frombuffer(archive, dtype=np.uint8)
    pieces = [a[s:e] for s, e in blocks]
    cat = np.concatenate(pieces) if len(pieces) > 1 else pieces[0]
    pos = 0
    for i, pc in enumerate(pieces):
        ranges[i] = pos
        pos += pc.size
    ranges[len(blocks)] = pos
    data, _, _, _ = _ctx().decompress_blocks(cat, ranges)
    out += data.tobytes()
    return bytes(out)
