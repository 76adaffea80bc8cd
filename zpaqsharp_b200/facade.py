"""The reference's streaming classes on top of the batch C ABI (SURVEY.md 8b, "streaming facade"): `Compressor`
(Compressor.cs:12-304), `Decompresser` (Decompresser.cs:13-204), `Reader` (Reader.cs:9-23) and `Writer` (Writer.cs:14-24) with
the reference's method names, argument meaning, call-order rules and error messages.  A segment is buffered on the host;
finished blocks are QUEUED and coded by the GPU a wave at a time through one batch call (`batch_blocks` of them are pending,
`flush()`, `close()` / leaving the `with` block) -- a block coded alone would wait for its own serial bit chain, ~2.5 s per MB
of mid.cfg, while a wave of 1600 takes the same time.  Everything written after a pending block is held back with it, so the
bytes reach the Writer in the reference's order and the archive is byte-identical to what the reference's classes write for
the same calls.  `batch_blocks=1` codes every block when it ends.  The Decompresser decodes a wave of the blocks ahead of the
one asked for in one call and serves `decompress(n)` from that.

libzpaq's encryption pieces under their libzpaq names: `AES_CTR(key, iv, ctx).encrypt(buf, n, offset)` (the keystream
computed and applied on the GPU), `stretchKey(in32, salt32)` and `scrypt(...)` (host), which StretchKey.cs:13-163 restates.
As in libzpaq they are building blocks: the caller writes the salt and encrypts the archive bytes behind it.

Deliberate limits of the device path, reported through `error()` like any other failure: one segment per block
(the batch ABI codes independent blocks; SURVEY.md 8f lists multi-segment blocks as a later step).  Nothing here touches
the oracle: without the CUDA library every call that needs the codec raises."""
from __future__ import annotations

import hashlib

import numpy as np

from . import libzpaq as z

TAG = bytes([0x37, 0x6B, 0x53, 0x74, 0xA0, 0x31, 0x83, 0xD3, 0x8C, 0xB2, 0x28, 0xB0, 0xD3])     # Compressor.cs:25-43


def error(msg: str):
    """LibZPAQ.error (LibZPAQ.cs:22-24): does not return."""
    raise z.ZpaqError(z.E_ARG, msg)


class Reader:
    """Reader.cs:9-23: get() returns a byte or -1; read(n) returns up to n bytes (default: by get())."""

    def get(self) -> int:
        raise NotImplementedError

    def read(self, n: int) -> bytes:
        out = bytearray()
        while len(out) < n:
            c = self.get()
            if c < 0:
                break
            out.append(c)
        return bytes(out)


class Writer:
    """Writer.cs:14-24: put(c) writes one byte; write(buf) writes many (default: by put())."""

    def put(self, c: int):
        raise NotImplementedError

    def write(self, buf: bytes):
        for c in buf:
            self.put(c)


class BytesReader(Reader):
    def __init__(self, data: bytes):
        self._d, self._i = memoryview(data), 0

    def get(self) -> int:
        if self._i >= len(self._d):
            return -1
        self._i += 1
        return self._d[self._i - 1]

    def read(self, n: int) -> bytes:
        b = bytes(self._d[self._i:self._i + n])
        self._i += len(b)
        return b


class BytesWriter(Writer):
    """Collects the bytes; reading them (`getvalue`) first makes the Compressors writing here code what they still hold."""

    def __init__(self):
        self.buf = bytearray()
        self._producers: list = []

    def put(self, c: int):
        self.buf.append(c & 255)

    def write(self, buf: bytes):
        self.buf += buf

    def getvalue(self) -> bytes:
        for p in list(self._producers):
            p.flush()
        return bytes(self.buf)


INIT, BLOCK1, SEG1, BLOCK2, SEG2 = range(5)            # Compressor.cs:314-322


class _Pending:
    """A finished block waiting for the GPU: what goes between its segment header and its end-of-block byte."""
    __slots__ = ("hdr", "pcomp", "data", "dosha1", "caller_sha1", "keep_sha1", "body")

    def __init__(self, hdr, pcomp, data, dosha1, caller_sha1, keep_sha1):
        self.hdr, self.pcomp, self.data, self.dosha1 = hdr, pcomp, data, dosha1
        self.caller_sha1, self.keep_sha1, self.body = caller_sha1, keep_sha1, None


class Compressor:
    """Compressor.cs:12-304.  Call order as in the reference: [writeTag] startBlock startSegment [postProcess]
    compress* endSegment endBlock.  `flush()` (or `close()`, or leaving a `with` block) codes what is still queued."""

    def __init__(self, ctx: z.Context | None = None, batch_blocks: int | None = None):
        self._ctx = ctx
        self._out: Writer | None = None
        self._in: Reader | None = None
        self._state = INIT
        self._verify = False
        self._hdr = b""
        self._pz = b""                 # PCOMP from startBlock(config, args)
        self._pcomp = b""              # PCOMP that goes into the first segment
        self._seg = bytearray()
        self._filename = self._comment = b""
        self._sha1 = b""
        self._last = b""
        self._batch = batch_blocks     # None: one resident wave of the model (estimated from its state size)
        self._queue: list = []         # bytes and _Pending items, in output order, from the first pending block on
        self._npending = 0

    # -- plumbing
    def _c(self) -> z.Context:
        if self._ctx is None:
            self._ctx = z._ctx()
        return self._ctx

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def close(self):
        self.flush()

    def _emit(self, b: bytes):
        """Bytes for the Writer: at once when no block is pending in front of them."""
        if self._queue:
            self._queue.append(bytes(b))
        else:
            self._out.write(b)

    def _wave(self, p: _Pending) -> int:
        if self._batch is not None:
            return max(1, self._batch)
        state = z.device_state_bytes(p.hdr)
        return max(1, min(148 * 16, int(150e9 // (state + 6 * max(len(p.data), 1 << 16)))))

    def flush(self):
        """Code every queued block (one batch call per model) and hand the held-back bytes to the Writer in order."""
        if not self._queue:
            return
        groups: dict = {}
        for it in self._queue:
            if isinstance(it, _Pending):
                groups.setdefault((it.hdr, it.pcomp, it.dosha1), []).append(it)
        for (hdr, pcomp, dosha1), items in groups.items():
            data = b"".join(it.data for it in items)
            offs = np.concatenate([[0], np.cumsum([len(it.data) for it in items])]).astype(np.uint64)
            arc, ooff = self._c().compress_blocks_model(data, offs, hdr, pcomp, [0] * 9, None, None, dosha1, False)
            for i, it in enumerate(items):
                a = arc[int(ooff[i]):int(ooff[i + 1])].tobytes()
                # what the library wrote in front of the coded bytes: "zPQ" level 1, header, segment header with its default comment
                skip = 5 + len(hdr) + 1 + 1 + len(str(len(it.data))) + 1 + 1
                assert a[:3] == b"zPQ" and a[-1] == 255
                body = a[skip:-1]
                if not dosha1:
                    assert body[-5:] == b"\x00\x00\x00\x00\xfe"
                    if it.caller_sha1 is not None:
                        body = body[:-1] + b"\xfd" + bytes(it.caller_sha1[:20])
                else:
                    assert body[-25:-20] == b"\x00\x00\x00\x00\xfd"
                    if not it.keep_sha1:
                        body = body[:-21] + b"\xfe"
                it.body = body
        q, self._queue, self._npending = self._queue, [], 0
        for it in q:
            self._out.write(it.body if isinstance(it, _Pending) else it)

    def setOutput(self, out: Writer):                  # Compressor.cs:20 (spelled `ssetOutput` there)
        self.flush()
        self._out = out
        prod = getattr(out, "_producers", None)
        if isinstance(prod, list) and self not in prod:
            prod.append(self)                          # a Writer that can be read back asks for the queued blocks first

    ssetOutput = setOutput

    def setInput(self, i: Reader):                     # Compressor.cs:148-151
        self._in = i

    def setVerify(self, v: bool):                      # Compressor.cs:118-121: the device always hashes what it codes
        self._verify = bool(v)

    # -- block
    def writeTag(self):                                # Compressor.cs:27-43
        assert self._state == INIT
        self._emit(TAG)

    def startBlock(self, model, args=None, pcomp_cmd: Writer | None = None):
        """startBlock(int level) / startBlock(hcomp bytes) / startBlock(config text, args) -- Compressor.cs:45-116."""
        assert self._state == INIT
        self._pz = b""
        if isinstance(model, int):
            if model < 1:
                error("compression level must be at least 1")
            if model > 3:
                error("compression level too high")
            hdr = z.builtin_model(model)
        elif isinstance(model, (bytes, bytearray, memoryview)):
            hdr = bytes(model)
        else:
            hdr, pz = z.compile_config(model if isinstance(model, str) else bytes(model).decode("latin-1"), args)
            self._pz = bytes(pz)                       # (the PCOMP command text before ";" is not kept by the library)
        self._hdr = bytes(hdr)
        if len(self._hdr) <= 6:
            error("invalid block header")
        self._emit(b"zPQ" + bytes([1 + (self._hdr[6] == 0), 1]) + self._hdr)      # Compressor.cs:91-96
        self._state = BLOCK1

    def hcomp(self, out2: Writer):                     # Compressor.cs:123-126
        out2.write(self._hdr)

    def pcomp(self, out2: Writer) -> bool:             # Compressor.cs:128-131
        if not self._pz:
            return False
        out2.write(bytes([len(self._pz) & 255, len(self._pz) >> 8]) + self._pz)
        return True

    # -- segment
    def startSegment(self, filename: str | bytes | None = None, comment: str | bytes | None = None):
        assert self._state in (BLOCK1, BLOCK2)
        if self._state == BLOCK2:
            error("the device path codes one segment per block")
        enc = lambda s: b"" if s is None else (s.encode() if isinstance(s, str) else bytes(s))
        self._filename, self._comment = enc(filename), enc(comment)
        self._emit(b"\x01" + self._filename + b"\x00" + self._comment + b"\x00\x00")   # Compressor.cs:133-146
        self._seg = bytearray()
        self._pcomp = b""
        self._state = SEG1

    def postProcess(self, pcomp: bytes | None = None, length: int = 0):
        """Compressor.cs:156-190: which PCOMP program the first segment starts with (none: a 0 byte)."""
        if self._state == SEG2:
            return
        assert self._state == SEG1
        if pcomp is None:
            self._pcomp = self._pz
        elif length == 0:
            n = pcomp[0] + 256 * pcomp[1]
            self._pcomp = bytes(pcomp[2:2 + n])
        else:
            self._pcomp = bytes(pcomp[:length])
        self._state = SEG2

    def compress(self, n: int = -1) -> bool:
        """Compressor.cs:193-221: take n bytes (all if n < 0) from the Reader; True until the input is exhausted."""
        if self._state == SEG1:
            self.postProcess()
        assert self._state == SEG2
        BUFSIZE = 1 << 20
        while n:
            nbuf = BUFSIZE if n < 0 or n >= BUFSIZE else n
            buf = self._in.read(nbuf)
            if len(buf) > nbuf:
                error("invalid read size")
            if not buf:
                return False
            if n >= 0:
                n -= len(buf)
            self._seg += buf
        return True

    def _enqueue(self, dosha1: bool, caller_sha1, keep_sha1: bool):
        p = _Pending(self._hdr, self._pcomp, bytes(self._seg), dosha1, caller_sha1, keep_sha1)
        self._last = p.data
        self._sha1 = b""
        self._queue.append(p)
        self._npending += 1
        self._state = BLOCK2
        return p

    def endSegment(self, sha1string: bytes | None = None):
        """Compressor.cs:224-249: end of data marker, then the caller's SHA-1 (253 + 20 bytes) or 254."""
        if self._state == SEG1:
            self.postProcess()
        assert self._state == SEG2
        self._enqueue(False, sha1string, False)

    def endSegmentChecksum(self, dosha1: bool = True):
        """Compressor.cs:251-281: as endSegment with the SHA-1 of what was coded (the device hashes the block for the trailer).
        Returns (sha1 or None, size) -- the reference returns the hash and writes the size through a pointer."""
        if self._state == SEG1:
            self.postProcess()
        assert self._state == SEG2
        self._enqueue(True, None, bool(self._verify and dosha1))
        return (self.getChecksum() if self._verify else None), len(self._seg)

    def getSize(self) -> int:                          # Compressor.cs:283-286
        return len(self._seg)

    def getChecksum(self) -> bytes:                    # Compressor.cs:288-291
        if not self._sha1:
            self._sha1 = hashlib.sha1(self._last).digest()
        return self._sha1

    def endBlock(self):                                # Compressor.cs:294-299
        assert self._state == BLOCK2
        self._emit(b"\xff")
        self._state = INIT
        if self._npending and self._npending >= self._wave(next(it for it in self._queue if isinstance(it, _Pending))):
            self.flush()


BLOCK, FILENAME, COMMENT, DATA, SEGEND = range(5)      # Decompresser.cs:206-213
FIRSTSEG, SEG, SKIP = range(3)                          # Decompresser.cs:214-219


class Decompresser:
    """Decompresser.cs:13-204.  findBlock reads the archive block from the Reader up to its end-of-block byte; the GPU
    decodes it when decompress() is first called."""

    def __init__(self, ctx: z.Context | None = None, batch_blocks: int | None = None):
        self._ctx = ctx
        self._batch = batch_blocks    # blocks decoded per GPU call (None: up to 2368 blocks / 2 GB of archive ahead)
        self._cache: dict = {}        # block index -> (restored bytes, sha1 status), decoded ahead
        self._in: Reader | None = None
        self._out: Writer | None = None
        self._state, self._dstate = BLOCK, FIRSTSEG
        self._arc = b""               # everything the Reader held, read once
        self._blocks: list = []       # [(start of "zPQ", one past the 255)], found once
        self._pos = 0
        self._blk = b""               # the current block from "zPQ" to its 255
        self._hdr = b""
        self._p = 0                   # parse position inside the block
        self._data: bytes | None = None
        self._dpos = 0
        self._sha_status = 0

    def _c(self) -> z.Context:
        if self._ctx is None:
            self._ctx = z._ctx()
        return self._ctx

    def setInput(self, i: Reader):                     # Decompresser.cs:22-25
        self._in = i
        self._arc, self._pos, self._blocks, self._next = b"", 0, [], 0
        self._cache = {}

    def setOutput(self, out: Writer | None):           # Decompresser.cs:113-116
        self._out = out

    def setSHA1(self, sha1ptr):                        # Decompresser.cs:118-121: the device verifies stored hashes itself
        self._sha1ptr = sha1ptr

    def _slurp(self):
        if not self._arc and self._in is not None:
            chunks = []
            while True:
                b = self._in.read(1 << 20)
                if not b:
                    break
                chunks.append(b)
            self._arc = b"".join(chunks)
            self._blocks = z.find_blocks(self._arc) if self._arc else []
            self._next = 0

    def findBlock(self, memptr: list | None = None) -> bool:
        """Decompresser.cs:29-58: scan for the locator tag, check level / type, read the header."""
        assert self._state == BLOCK
        self._slurp()
        if self._next >= len(self._blocks):
            self._pos = len(self._arc)
            return False
        s, e = self._blocks[self._next]
        self._next += 1
        i = 0
        blk = self._arc[s:e]
        if blk[3] not in (1, 2):
            error("unsupported ZPAQ level")
        if blk[4] != 1:
            error("unsupported ZPAQL type")
        hsize = blk[5] + 256 * blk[6]
        self._hdr = blk[5:5 + hsize + 2]
        if blk[3] == 1 and len(self._hdr) > 6 and self._hdr[6] == 0:
            error("ZPAQ level 1 requires at least 1 component")
        if memptr is not None:
            memptr[:] = [z.block_memory(self._hdr)]
        self._blk, self._p, self._pos = blk, 5 + hsize + 2, i + e
        self._data, self._dpos = None, 0
        self._state, self._dstate = FILENAME, FIRSTSEG
        return True

    def hcomp(self, out2: Writer):                     # Decompresser.cs:60-63
        out2.write(self._hdr)

    def _get(self) -> int:
        if self._p >= len(self._blk):
            return -1
        self._p += 1
        return self._blk[self._p - 1]

    def findFilename(self, filename: Writer | None = None) -> bool:
        """Decompresser.cs:65-93: a segment (1, name, 0) or the end of the block (255)."""
        assert self._state == FILENAME
        c = self._get()
        if c == 1:
            if self._dstate != FIRSTSEG:
                error("the device path decodes one segment per block")
            while True:
                c = self._get()
                if c == -1:
                    error("unexpected EOF")
                if c == 0:
                    self._state = COMMENT
                    return True
                if filename is not None:
                    filename.put(c)
        elif c == 255:
            self._state = BLOCK
            return False
        else:
            error("missing segment or end of block")
        return False

    def readComment(self, comment: Writer | None = None):
        """Decompresser.cs:95-111."""
        assert self._state == COMMENT
        self._state = DATA
        while True:
            c = self._get()
            if c == -1:
                error("unexpected EOF")
            if c == 0:
                break
            if comment is not None:
                comment.put(c)
        if self._get() != 0:
            error("missing reserved byte")

    def _decode(self):
        """The current block's restored bytes: decoded together with a wave of the blocks behind it (one GPU call)."""
        if self._data is None:
            cur = self._next - 1
            if cur not in self._cache:
                self._cache = {}
                limit = self._batch if self._batch is not None else 148 * 16
                hi, nbytes = cur, 0
                while hi < len(self._blocks) and hi - cur < max(1, limit) and nbytes < (2 << 30):
                    nbytes += self._blocks[hi][1] - self._blocks[hi][0]
                    hi += 1
                a = np.frombuffer(self._arc, dtype=np.uint8)
                pieces = [a[s:e] for s, e in self._blocks[cur:hi]]
                cat = np.concatenate(pieces) if len(pieces) > 1 else pieces[0]
                offs = np.concatenate([[0], np.cumsum([p.size for p in pieces])]).astype(np.uint64)
                try:
                    out, ooff, sha, _ = self._c().decompress_blocks(cat, offs)
                except z.ZpaqError:
                    if hi - cur == 1:
                        raise
                    # a damaged block somewhere ahead must not fail this one: decode it alone
                    out, ooff, sha, _ = self._c().decompress_blocks(pieces[0], offs[:2])
                    hi = cur + 1
                for k in range(hi - cur):
                    self._cache[cur + k] = (out[int(ooff[k]):int(ooff[k + 1])].tobytes(), int(sha[k]))
            self._data, self._sha_status = self._cache.pop(cur)
            self._dstate = SEG

    def decompress(self, n: int = -1) -> bool:
        """Decompresser.cs:123-155: n bytes (all if n < 0) to the Writer; False once the segment is exhausted."""
        assert self._state == DATA
        if self._dstate == SKIP:
            error("decompression after skipped segment")
        self._decode()
        left = len(self._data) - self._dpos
        take = left if n < 0 else min(n, left)
        if self._out is not None and take:
            self._out.write(self._data[self._dpos:self._dpos + take])
        self._dpos += take
        if n < 0 or take < n:                          # the end-of-segment marker was reached
            self._state = SEGEND
            return False
        return True

    def readSegmentEnd(self, sha1string: bytearray | None = None):
        """Decompresser.cs:160-194: 254, or 253 + the stored SHA-1; sha1string[0] = 1 and the 20 bytes, or 0."""
        assert self._state in (DATA, SEGEND)
        if self._state == DATA:
            self._dstate = SKIP
        b = self._blk
        if len(b) >= 27 and b[-26:-21] == b"\x00\x00\x00\x00\xfd":
            if sha1string is not None:
                sha1string[0:21] = b"\x01" + b[-21:-1]
            self._p = len(b) - 1
        elif len(b) >= 7 and b[-6:-1] == b"\x00\x00\x00\x00\xfe":
            if sha1string is not None:
                sha1string[0:1] = b"\x00"
            self._p = len(b) - 1
        else:
            error("missing end of segment marker")
        self._state = FILENAME

    def sha1_verified(self) -> int:
        """Device-side check of the stored SHA-1 of the segment just decoded: 0 none stored, 1 match, 2 mismatch."""
        return self._sha_status

    def buffered(self) -> int:                         # Decompresser.cs:201-204
        return len(self._arc) - self._pos


# ---- encryption (libzpaq 7.12 AES_CTR, stretchKey, scrypt) --------------------------------------------------------------
class AES_CTR:
    """libzpaq AES_CTR(key, keylen, iv): encrypt(buf, n, offset) XORs buf[0..n) with the keystream from stream byte offset
    (block j = AES(iv[0..7] || big-endian j)); decrypting is the same call.  key is 16, 24 or 32 bytes; iv 8 bytes or None."""

    def __init__(self, key: bytes, iv: bytes | None = None, ctx: z.Context | None = None):
        if len(key) not in (16, 24, 32):
            error("AES key length must be 16, 24 or 32 bytes")
        self._key, self._iv, self._ctx = bytes(key), iv, ctx

    def encrypt(self, buf, n: int, offset: int):
        """In place on the first n bytes of a writable buffer (bytearray, numpy uint8, ...)."""
        a = buf if isinstance(buf, np.ndarray) else np.frombuffer(buf, dtype=np.uint8)
        if n < 0 or n > a.size:
            error("AES_CTR.encrypt: n is outside the buffer")
        (self._ctx or z._ctx()).aes_ctr(a[:n], self._key, self._iv, offset)


def stretchKey(in32: bytes, salt32: bytes) -> bytes:
    """libzpaq stretchKey(out, in, salt): scrypt(in, salt, 16384, 8, 1, 32); in32 is SHA-256 of the password."""
    return z.stretch_key(in32, salt32)


def scrypt(pw: bytes, salt: bytes, n: int, r: int, p: int, dklen: int) -> bytes:
    """libzpaq scrypt(pw, pwlen, salt, saltlen, n, r, p, out, outlen) (RFC 7914)."""
    return z.scrypt(pw, salt, n, r, p, dklen)
