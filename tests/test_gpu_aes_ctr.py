"""GPU: libzpaq 7.12's AES_CTR::encrypt(buf, n, offset) (zpq_aes_ctr on host buffers, zpq_aes_ctr_dev on device buffers)
against the `cryptography` package's AES-CTR, and an encrypted archive (salt || AES-CTR(archive), key from stretchKey) taken
apart and decoded again.  The two-device test is skipped on a single-GPU box, like tests/test_gpu_multi.py."""
import ctypes as C
import hashlib
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cryptography = pytest.importorskip("cryptography")
from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes  # noqa: E402


def ref_ctr(data: bytes, key: bytes, iv, offset: int) -> bytes:
    """libzpaq's layout: keystream block j = AES(iv[0..7] || BE64(j)); byte offset + k uses block (offset + k) / 16."""
    e = Cipher(algorithms.AES(key), modes.CTR((iv or bytes(8)) + (offset // 16).to_bytes(8, "big"))).encryptor()
    e.update(bytes(offset % 16))
    return e.update(data)


def _ndev():
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for line in out.splitlines() if line.startswith("GPU "))
    except Exception:
        return 0


def test_every_alignment_offset_and_length_host_and_device(gpu_ctx):
    import torch
    rng = random.Random(1)
    key, iv = rng.randbytes(32), rng.randbytes(8)
    lengths = [0, 1, 15, 16, 17, 31, 33, 80]
    host = np.zeros(160, dtype=np.uint8)
    dev = torch.zeros(160, dtype=torch.uint8, device="cuda")
    bad = []
    for mis in range(16):
        for r in range(16):
            offset = 16 * 1000003 + r
            for n in lengths:
                plain = rng.randbytes(n)
                want = ref_ctr(plain, key, iv, offset)
                h = host[mis:mis + n]
                h[:] = np.frombuffer(plain, dtype=np.uint8)
                gpu_ctx.aes_ctr(h, key, iv, offset)
                if h.tobytes() != want:
                    bad.append(("host", mis, r, n))
                d = dev[mis:mis + n]
                d.copy_(torch.frombuffer(bytearray(plain), dtype=torch.uint8) if n else torch.empty(0, dtype=torch.uint8))
                torch.cuda.synchronize()                 # torch's copy runs on its own stream, the library on the context's
                gpu_ctx.aes_ctr_dev(d.data_ptr(), n, key, iv, offset)
                torch.cuda.synchronize()
                if bytes(d.cpu().numpy().tobytes()) != want:
                    bad.append(("dev", mis, r, n))
                # the bytes around the range stay as they were
                assert not host[:mis].any() and not host[mis + n:].any()
                host[:] = 0
                assert int(dev[:mis].count_nonzero()) == 0 and int(dev[mis + n:].count_nonzero()) == 0
                dev.zero_()
    assert not bad, bad[:20]


@pytest.mark.parametrize("keylen", [16, 24, 32])
def test_key_lengths_null_iv_and_high_counters(gpu_ctx, keylen):
    import torch
    rng = random.Random(keylen)
    key = rng.randbytes(keylen)
    for offset in [0, 7, (1 << 40) + 7, (1 << 63) + 5, (1 << 64) - 1 - 5000]:
        for iv in [None, rng.randbytes(8)]:
            plain = rng.randbytes(5000)
            want = ref_ctr(plain, key, iv, offset)
            assert bytes(gpu_ctx.aes_ctr(bytearray(plain), key, iv, offset)) == want, (offset, iv)
            d = torch.frombuffer(bytearray(plain), dtype=torch.uint8).cuda()
            torch.cuda.synchronize()
            gpu_ctx.aes_ctr_dev(d.data_ptr(), d.numel(), key, iv, offset)
            assert d.cpu().numpy().tobytes() == want, (offset, iv)
    st = gpu_ctx.stats()
    assert st.kernel.decode() == "aes_ctr/%d" % (8 * keylen) and st.launches == 1 and st.kernel_ms > 0


def test_large_host_buffer_goes_through_several_chunks(gpu_ctx):
    n = 3 * (1 << 29) + 12345                                    # 1.5 GiB and a bit: two 1 GiB chunks
    rng = np.random.default_rng(3)
    plain = rng.integers(0, 256, n, dtype=np.uint8)
    key, iv, offset = bytes(range(32)), bytes(range(8, 16)), 123456789
    want = np.frombuffer(ref_ctr(memoryview(plain), key, iv, offset), dtype=np.uint8)
    buf = plain.copy()
    del plain
    gpu_ctx.aes_ctr(buf, key, iv, offset)
    assert np.array_equal(buf, want)
    st = gpu_ctx.stats()
    assert st.launches == 2 and st.h2d_bytes == n and st.d2h_bytes == n and st.kernel.decode() == "aes_ctr/256"
    assert st.h2d_ms > 0 and st.d2h_ms > 0 and st.total_ms >= st.kernel_ms


def test_split_calls_equal_one_call_and_twice_is_identity(gpu_ctx):
    rng = random.Random(9)
    key, iv = rng.randbytes(24), rng.randbytes(8)
    plain = rng.randbytes(100003)
    a, c = 77, 100003
    whole = bytes(gpu_ctx.aes_ctr(bytearray(plain[:c]), key, iv, a))
    for b in [77, 78, 93, 5000, 5001, 65536 + 3, 99999]:
        left = gpu_ctx.aes_ctr(bytearray(plain[:b - a]), key, iv, a)
        right = gpu_ctx.aes_ctr(bytearray(plain[b - a:c]), key, iv, b)
        assert bytes(left) + bytes(right) == whole, b
    assert whole == ref_ctr(plain[:c], key, iv, a)
    assert bytes(gpu_ctx.aes_ctr(bytearray(whole), key, iv, a)) == plain[:c]


def test_argument_errors_with_a_context(gpu_ctx, zlib_):
    L = zlib_.load()
    h = gpu_ctx._h
    buf = (C.c_uint8 * 64)()
    for call in (L.zpq_aes_ctr, L.zpq_aes_ctr_dev):
        for keylen in (0, 8, 15, 17, 31, 33, 64):
            assert call(h, bytes(64), keylen, None, buf, 16, 0) == zlib_.E_ARG, keylen
        assert call(h, None, 16, None, buf, 16, 0) == zlib_.E_ARG
        assert call(h, bytes(16), 16, None, None, 16, 0) == zlib_.E_ARG
        assert call(h, bytes(16), 16, None, None, 0, 0) == 0                      # n = 0: nothing to do
    assert L.zpq_aes_ctr(h, bytes(16), 16, None, buf, 1, (1 << 64) - 1) == zlib_.E_ARG   # offset + n past 2^64 - 1
    assert L.zpq_aes_ctr(h, bytes(16), 16, None, buf, 64, (1 << 64) - 64) == zlib_.E_ARG
    assert L.zpq_aes_ctr(h, bytes(16), 16, None, buf, 63, (1 << 64) - 64) == 0           # ends at 2^64 - 1
    assert bytes(buf)[:63] == ref_ctr(bytes(63), bytes(16), None, (1 << 64) - 64)
    with pytest.raises(zlib_.ZpaqError) as e:
        gpu_ctx.aes_ctr(bytearray(8), bytes(20))
    assert e.value.code == zlib_.E_ARG
    with pytest.raises(TypeError):
        gpu_ctx.aes_ctr(b"read-only", bytes(16))


def test_encrypted_archive_decrypts_and_decodes(gpu_ctx, zlib_, oracle):
    from tools import synth
    rng = random.Random(2024)
    data = synth.blocks("mixed", 77, 12, 20000).tobytes()
    cuts = sorted(set([0, len(data)] + [rng.randrange(1, len(data)) for _ in range(11)]))
    offs = np.asarray(cuts, dtype=np.uint64)
    half = len(cuts) // 2
    arc_mid, _ = gpu_ctx.compress_blocks_level(data, offs[:half + 1], 2)                       # mid.cfg
    lz_offs = offs[half:] - offs[half]
    arc_lz, lz_ooff = gpu_ctx.compress_blocks(data[cuts[half]:], lz_offs, "x0,1,4,0,7,21,1")    # bit-packed LZ77
    assert arc_lz[:int(lz_ooff[1])].tobytes() == oracle.compress_block(data[cuts[half]:cuts[half + 1]], "x0,1,4,0,7,21,1")
    archive = arc_mid.tobytes() + arc_lz.tobytes()

    password, salt = b"correct horse battery staple", rng.randbytes(32)
    key = zlib_.stretch_key(hashlib.sha256(password).digest(), salt)
    assert key == hashlib.scrypt(hashlib.sha256(password).digest(), salt=salt, n=16384, r=8, p=1, dklen=32)
    enc = salt + bytes(gpu_ctx.aes_ctr(bytearray(archive), key, salt[:8], 32))
    assert enc[32:] == ref_ctr(archive, key, salt[:8], 32)

    body = gpu_ctx.aes_ctr(bytearray(enc[32:]), key, salt[:8], 32)
    assert bytes(body) == archive
    blocks = zlib_.find_blocks(body)
    assert len(blocks) == len(cuts) - 1
    a = np.frombuffer(body, dtype=np.uint8)
    cat = np.concatenate([a[s:e] for s, e in blocks])
    ranges = np.cumsum([0] + [e - s for s, e in blocks]).astype(np.uint64)
    out, _, sha, bst = gpu_ctx.decompress_blocks(cat, ranges)
    assert out.tobytes() == data and set(sha.tolist()) == {1} and not bst.any()


@pytest.mark.skipif(_ndev() < 2, reason="needs two GPUs")
def test_context_on_all_devices_matches_one_device(zlib_):
    nd = _ndev()
    rng = np.random.default_rng(11)
    n, offset = 50_000_017, 987_654_321_011
    plain = rng.integers(0, 256, n, dtype=np.uint8)
    key, iv = bytes(range(100, 132)), bytes(range(8))
    with zlib_.Context([0]) as one, zlib_.Context(list(range(nd))) as many:
        a = one.aes_ctr(plain.copy(), key, iv, offset)
        b = many.aes_ctr(plain.copy(), key, iv, offset)
    assert np.array_equal(a, b)
    assert a.tobytes() == ref_ctr(plain.tobytes(), key, iv, offset)


def test_facade_aes_ctr_and_stretch_key(gpu_ctx):
    from zpaqsharp_b200 import facade as f
    rng = random.Random(31)
    key, iv = rng.randbytes(16), rng.randbytes(8)
    buf = bytearray(rng.randbytes(1000))
    plain = bytes(buf)
    f.AES_CTR(key, iv, gpu_ctx).encrypt(buf, 600, 12345)                 # the first n bytes only
    assert bytes(buf[:600]) == ref_ctr(plain[:600], key, iv, 12345) and buf[600:] == plain[600:]
    f.AES_CTR(key, iv, gpu_ctx).encrypt(buf, 600, 12345)
    assert bytes(buf) == plain
    in32, salt = hashlib.sha256(b"pw").digest(), rng.randbytes(32)
    assert f.stretchKey(in32, salt) == hashlib.scrypt(in32, salt=salt, n=16384, r=8, p=1, dklen=32)
    assert f.scrypt(b"pw", b"salt", 16, 1, 1, 20) == hashlib.scrypt(b"pw", salt=b"salt", n=16, r=1, p=1, dklen=20)
    with pytest.raises(Exception):
        f.AES_CTR(bytes(10))
