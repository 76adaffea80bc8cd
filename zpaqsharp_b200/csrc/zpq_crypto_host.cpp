// zpq_crypto_host.cpp -- the host half of libzpaq 7.12's encryption: the AES key schedule, SHA-256 (FIPS 180-4),
// HMAC / PBKDF2-HMAC-SHA256 and scrypt (RFC 7914), which libzpaq's stretchKey calls (StretchKey.cs:13-163 restates it).
//
// Key derivation stays on the host: stretchKey is one scrypt per archive, a single serial ROMix chain over 16 MiB
// (n = 16384, r = 8, p = 1) with no independent work to spread over a device.
#include <algorithm>
#include <cstring>
#include <utility>
#include <vector>

#include "zpq_crypto.h"
#include "zpq_host.h"

namespace zpq {

static const uint8_t kSbox[256] = ZPQ_AES_SBOX;

void secure_zero(void* p, size_t n) {
  volatile uint8_t* q = static_cast<volatile uint8_t*>(p);
  while (n--) *q++ = 0;
}

// ---- AES key schedule (FIPS-197 5.2) --------------------------------------------------------------------------------
void aes_expand_key(const uint8_t* key, int keylen, AesKey& out) {
  const int nk = keylen / 4;
  out.rounds = nk + 6;
  const int words = 4 * (out.rounds + 1);
  uint32_t rcon = 1;
  for (int i = 0; i < 60; ++i) out.rk[i] = 0;
  for (int i = 0; i < nk; ++i)
    out.rk[i] = (uint32_t)key[4 * i] << 24 | (uint32_t)key[4 * i + 1] << 16 | (uint32_t)key[4 * i + 2] << 8 | key[4 * i + 3];
  auto sub = [](uint32_t w) {
    return (uint32_t)kSbox[w >> 24] << 24 | (uint32_t)kSbox[(w >> 16) & 255] << 16 | (uint32_t)kSbox[(w >> 8) & 255] << 8 | kSbox[w & 255];
  };
  for (int i = nk; i < words; ++i) {
    uint32_t t = out.rk[i - 1];
    if (i % nk == 0) {
      t = sub(t << 8 | t >> 24) ^ rcon << 24;
      rcon = (rcon << 1) ^ ((rcon >> 7) * 0x11b);
    } else if (nk > 6 && i % nk == 4) {
      t = sub(t);
    }
    out.rk[i] = out.rk[i - nk] ^ t;
  }
}

// ---- SHA-256 (FIPS 180-4) --------------------------------------------------------------------------------------------
namespace {

const uint32_t kK256[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01,
    0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc,
    0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147,
    0x06ca6351, 0x14292967, 0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85,
    0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08,
    0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208,
    0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};

inline uint32_t ror(uint32_t x, int k) { return x >> k | x << (32 - k); }

struct Sha256 {
  uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
  uint8_t buf[64];
  uint64_t len = 0;   // bytes hashed so far

  void block(const uint8_t* p) {
    uint32_t w[64];
    for (int i = 0; i < 16; ++i) w[i] = (uint32_t)p[4 * i] << 24 | (uint32_t)p[4 * i + 1] << 16 | (uint32_t)p[4 * i + 2] << 8 | p[4 * i + 3];
    for (int i = 16; i < 64; ++i) {
      const uint32_t s0 = ror(w[i - 15], 7) ^ ror(w[i - 15], 18) ^ (w[i - 15] >> 3);
      const uint32_t s1 = ror(w[i - 2], 17) ^ ror(w[i - 2], 19) ^ (w[i - 2] >> 10);
      w[i] = w[i - 16] + s0 + w[i - 7] + s1;
    }
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], k = h[7];
    for (int i = 0; i < 64; ++i) {
      const uint32_t t1 = k + (ror(e, 6) ^ ror(e, 11) ^ ror(e, 25)) + ((e & f) ^ (~e & g)) + kK256[i] + w[i];
      const uint32_t t2 = (ror(a, 2) ^ ror(a, 13) ^ ror(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
      k = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += k;
    secure_zero(w, sizeof w);
  }
  void put(const uint8_t* p, uint64_t n) {
    while (n) {
      const uint32_t used = (uint32_t)(len % 64);
      if (used == 0 && n >= 64) { block(p); p += 64; n -= 64; len += 64; continue; }
      const uint32_t take = (uint32_t)std::min<uint64_t>(64 - used, n);
      memcpy(buf + used, p, take);
      p += take; n -= take; len += take;
      if (len % 64 == 0) block(buf);
    }
  }
  void finish(uint8_t out[32]) {
    const uint64_t bits = len * 8;
    const uint8_t pad = 0x80, zero = 0;
    put(&pad, 1);
    while (len % 64 != 56) put(&zero, 1);
    uint8_t be[8];
    for (int i = 0; i < 8; ++i) be[i] = (uint8_t)(bits >> (56 - 8 * i));
    put(be, 8);
    for (int i = 0; i < 8; ++i) for (int b = 0; b < 4; ++b) out[4 * i + b] = (uint8_t)(h[i] >> (24 - 8 * b));
  }
  ~Sha256() { secure_zero(h, sizeof h); secure_zero(buf, sizeof buf); }
};

void sha256(const uint8_t* p, uint64_t n, uint8_t out[32]) {
  Sha256 h;
  h.put(p, n);
  h.finish(out);
}

// HMAC-SHA256 (RFC 2104) with the key's inner and outer states computed once.
struct HmacSha256 {
  Sha256 inner, outer;
  HmacSha256(const uint8_t* key, uint64_t keylen) {
    uint8_t k[64] = {0}, pad[64];
    if (keylen > 64) sha256(key, keylen, k);   // a key longer than the block is hashed first
    else if (keylen) memcpy(k, key, keylen);
    for (int i = 0; i < 64; ++i) pad[i] = k[i] ^ 0x36;
    inner.put(pad, 64);
    for (int i = 0; i < 64; ++i) pad[i] = k[i] ^ 0x5c;
    outer.put(pad, 64);
    secure_zero(k, sizeof k); secure_zero(pad, sizeof pad);
  }
  // mac(prefix || msg)
  void mac(const uint8_t* msg, uint64_t n, const uint8_t* msg2, uint64_t n2, uint8_t out[32]) const {
    Sha256 i = inner, o = outer;
    uint8_t d[32];
    i.put(msg, n);
    if (n2) i.put(msg2, n2);
    i.finish(d);
    o.put(d, 32);
    o.finish(out);
    secure_zero(d, sizeof d);
  }
};

// ---- scrypt (RFC 7914) ------------------------------------------------------------------------------------------------
inline uint32_t rol(uint32_t x, int k) { return x << k | x >> (32 - k); }

void salsa20_8(uint32_t b[16]) {
  uint32_t x[16];
  memcpy(x, b, sizeof x);
  for (int i = 0; i < 8; i += 2) {
    x[4] ^= rol(x[0] + x[12], 7);   x[8] ^= rol(x[4] + x[0], 9);    x[12] ^= rol(x[8] + x[4], 13);   x[0] ^= rol(x[12] + x[8], 18);
    x[9] ^= rol(x[5] + x[1], 7);    x[13] ^= rol(x[9] + x[5], 9);   x[1] ^= rol(x[13] + x[9], 13);   x[5] ^= rol(x[1] + x[13], 18);
    x[14] ^= rol(x[10] + x[6], 7);  x[2] ^= rol(x[14] + x[10], 9);  x[6] ^= rol(x[2] + x[14], 13);   x[10] ^= rol(x[6] + x[2], 18);
    x[3] ^= rol(x[15] + x[11], 7);  x[7] ^= rol(x[3] + x[15], 9);   x[11] ^= rol(x[7] + x[3], 13);   x[15] ^= rol(x[11] + x[7], 18);
    x[1] ^= rol(x[0] + x[3], 7);    x[2] ^= rol(x[1] + x[0], 9);    x[3] ^= rol(x[2] + x[1], 13);    x[0] ^= rol(x[3] + x[2], 18);
    x[6] ^= rol(x[5] + x[4], 7);    x[7] ^= rol(x[6] + x[5], 9);    x[4] ^= rol(x[7] + x[6], 13);    x[5] ^= rol(x[4] + x[7], 18);
    x[11] ^= rol(x[10] + x[9], 7);  x[8] ^= rol(x[11] + x[10], 9);  x[9] ^= rol(x[8] + x[11], 13);   x[10] ^= rol(x[9] + x[8], 18);
    x[12] ^= rol(x[15] + x[14], 7); x[13] ^= rol(x[12] + x[15], 9); x[14] ^= rol(x[13] + x[12], 13); x[15] ^= rol(x[14] + x[13], 18);
  }
  for (int i = 0; i < 16; ++i) b[i] += x[i];
}

// scryptBlockMix: b (2r 64-byte blocks, as little-endian words) -> y; the even results go to the first half, the odd ones
// to the second.
void block_mix(const uint32_t* b, uint32_t* y, uint32_t r) {
  uint32_t x[16];
  memcpy(x, b + (2 * r - 1) * 16, sizeof x);
  for (uint32_t i = 0; i < 2 * r; ++i) {
    for (int t = 0; t < 16; ++t) x[t] ^= b[i * 16 + t];
    salsa20_8(x);
    memcpy(y + ((i & 1) * r + i / 2) * 16, x, sizeof x);
  }
}

// scryptROMix over one 128*r-byte chunk of B, in place; v holds n * 32 * r words, xy 64 * r.
void ro_mix(uint8_t* chunk, uint32_t r, uint64_t n, uint32_t* v, uint32_t* xy) {
  const uint64_t w = 32ull * r;
  uint32_t* x = xy;
  uint32_t* y = xy + w;
  for (uint64_t k = 0; k < w; ++k)
    x[k] = (uint32_t)chunk[4 * k] | (uint32_t)chunk[4 * k + 1] << 8 | (uint32_t)chunk[4 * k + 2] << 16 | (uint32_t)chunk[4 * k + 3] << 24;
  for (uint64_t i = 0; i < n; ++i) {
    memcpy(v + i * w, x, 4 * w);
    block_mix(x, y, r);
    std::swap(x, y);
  }
  for (uint64_t i = 0; i < n; ++i) {
    const uint32_t* last = x + (2 * r - 1) * 16;
    const uint64_t j = ((uint64_t)last[1] << 32 | last[0]) & (n - 1);     // Integerify
    for (uint64_t k = 0; k < w; ++k) x[k] ^= v[j * w + k];
    block_mix(x, y, r);
    std::swap(x, y);
  }
  for (uint64_t k = 0; k < w; ++k)
    for (int b = 0; b < 4; ++b) chunk[4 * k + b] = (uint8_t)(x[k] >> (8 * b));
}

void pbkdf2_sha256(const uint8_t* pw, uint64_t pwlen, const uint8_t* salt, uint64_t saltlen, uint64_t iters, uint8_t* out,
                   uint64_t outlen) {
  const HmacSha256 prf(pw, pwlen);
  uint8_t u[32], t[32], ctr[4];
  for (uint64_t blk = 1, done = 0; done < outlen; ++blk) {
    for (int b = 0; b < 4; ++b) ctr[b] = (uint8_t)(blk >> (24 - 8 * b));
    prf.mac(salt, saltlen, ctr, 4, u);
    memcpy(t, u, 32);
    for (uint64_t it = 1; it < iters; ++it) {
      prf.mac(u, 32, nullptr, 0, u);
      for (int b = 0; b < 32; ++b) t[b] ^= u[b];
    }
    const uint64_t take = std::min<uint64_t>(32, outlen - done);
    memcpy(out + done, t, take);
    done += take;
  }
  secure_zero(u, sizeof u); secure_zero(t, sizeof t);
}

}  // namespace

void scrypt(const uint8_t* pw, uint64_t pwlen, const uint8_t* salt, uint64_t saltlen, uint64_t n, uint32_t r, uint32_t p,
            uint8_t* out, uint64_t outlen) {
  if (n < 2 || (n & (n - 1)) || r == 0 || p == 0) throw Failure(ZPQ_E_ARG, "scrypt: n must be a power of two >= 2, r and p >= 1");
  const uint64_t chunk = 128ull * r;
  if ((uint64_t)p > ~0ull / chunk || n > ~0ull / chunk / 2) throw Failure(ZPQ_E_NOMEM, "scrypt: memory request too large");
  std::vector<uint8_t> b;
  std::vector<uint32_t> v, xy;
  try {
    b.resize(chunk * p);
    v.resize(n * 32ull * r);
    xy.resize(64ull * r);
  } catch (const std::exception&) {
    throw Failure(ZPQ_E_NOMEM, "scrypt: cannot allocate 128 * r * n bytes");
  }
  pbkdf2_sha256(pw, pwlen, salt, saltlen, 1, b.data(), b.size());
  for (uint32_t i = 0; i < p; ++i) ro_mix(b.data() + chunk * i, r, n, v.data(), xy.data());
  pbkdf2_sha256(pw, pwlen, b.data(), b.size(), 1, out, outlen);
  secure_zero(b.data(), b.size());
  secure_zero(v.data(), v.size() * 4);
  secure_zero(xy.data(), xy.size() * 4);
}

}  // namespace zpq
