"""Host key derivation of the encryption entry points (libzpaq 7.12's scrypt / stretchKey, StretchKey.cs:13-163) against
RFC 7914 and Python's hashlib, plus the argument checks of the AES-CTR entry points that fail before any device work."""
import ctypes as C
import hashlib
import random

import pytest

# RFC 7914 section 12, vectors 1-3 (vector 4 needs 1 GiB)
RFC7914 = [
    (b"", b"", 16, 1, 1, 64,
     "77d6576238657b203b19ca42c18a0497f16b4844e3074ae8dfdffa3fede21442fcd0069ded0948f8326a753a0fc81f17e8d3e0fb2e0d3628cf35e20c38d18906"),
    (b"password", b"NaCl", 1024, 8, 16, 64,
     "fdbabe1c9d3472007856e7190d01e9fe7c6ad7cbc8237830e77376634b3731622eaf30d92e22a3886ff109279d9830dac727afb94a83ee6d8360cbdfa2cc0640"),
    (b"pleaseletmein", b"SodiumChloride", 16384, 8, 1, 64,
     "7023bdcb3afd7348461c06cd81fd38ebfda8fbba904f8e3ea9b543f6545da1f2d5432955613f0fcf62d49705242a9af9e61e85dc0d651e40dfcf017b45575887"),
]


@pytest.mark.parametrize("pw,salt,n,r,p,dklen,hexout", RFC7914)
def test_scrypt_rfc7914_vectors(zlib_, pw, salt, n, r, p, dklen, hexout):
    assert zlib_.scrypt(pw, salt, n, r, p, dklen).hex() == hexout


def test_scrypt_matches_hashlib_on_random_parameters(zlib_):
    rng = random.Random(7914)
    for _ in range(50):
        pw = rng.randbytes(rng.randint(0, 200))            # past the 64-byte HMAC block: the hashed-key branch
        salt = rng.randbytes(rng.randint(0, 100))
        n = 1 << rng.randint(1, 10)
        r, p = rng.randint(1, 8), rng.randint(1, 3)
        dklen = rng.choice([1, 31, 32, 33, 64, 100])
        ref = hashlib.scrypt(pw, salt=salt, n=n, r=r, p=p, dklen=dklen)
        assert zlib_.scrypt(pw, salt, n, r, p, dklen) == ref, (len(pw), len(salt), n, r, p, dklen)


def test_stretch_key_is_scrypt_16384_8_1(zlib_):
    rng = random.Random(5)
    for _ in range(2):
        in32 = hashlib.sha256(rng.randbytes(rng.randint(0, 40))).digest()
        salt32 = rng.randbytes(32)
        assert zlib_.stretch_key(in32, salt32) == hashlib.scrypt(in32, salt=salt32, n=16384, r=8, p=1, dklen=32)


def test_scrypt_argument_errors(zlib_):
    L = zlib_.load()
    out = C.create_string_buffer(32)
    for n, r, p in [(0, 1, 1), (1, 1, 1), (3, 1, 1), (1000, 1, 1), (16, 0, 1), (16, 1, 0)]:
        assert L.zpq_scrypt(b"pw", 2, b"s", 1, n, r, p, out, 32) == zlib_.E_ARG, (n, r, p)
    assert L.zpq_scrypt(None, 2, b"s", 1, 16, 1, 1, out, 32) == zlib_.E_ARG
    assert L.zpq_scrypt(b"pw", 2, None, 1, 16, 1, 1, out, 32) == zlib_.E_ARG
    assert L.zpq_scrypt(b"pw", 2, b"s", 1, 16, 1, 1, None, 32) == zlib_.E_ARG
    assert L.zpq_scrypt(None, 0, None, 0, 16, 1, 1, None, 0) == 0              # nothing asked, nothing done
    assert L.zpq_scrypt(b"pw", 2, b"s", 1, 1 << 62, 8, 1, out, 32) == zlib_.E_NOMEM
    assert L.zpq_stretch_key(None, b"s" * 32, out) == zlib_.E_ARG
    with pytest.raises(zlib_.ZpaqError) as e:
        zlib_.scrypt(b"pw", b"salt", 6, 1, 1, 32)
    assert e.value.code == zlib_.E_ARG


def test_aes_ctr_refuses_a_null_context(zlib_):
    # the other argument errors (key length, null buffer, offset + n overflow) need a context: tests/test_gpu_aes_ctr.py
    L = zlib_.load()
    buf = (C.c_uint8 * 16)()
    for call in (L.zpq_aes_ctr, L.zpq_aes_ctr_dev):
        assert call(None, bytes(32), 32, None, buf, 16, 0) == zlib_.E_ARG
