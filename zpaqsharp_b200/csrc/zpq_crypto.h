// zpq_crypto.h -- encryption pieces of libzpaqb200 (not part of the C ABI): libzpaq 7.12's AES_CTR on the device
// (zpq_crypto.cu), its key schedule, SHA-256, PBKDF2-HMAC-SHA256 and scrypt on the host (zpq_crypto_host.cpp).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace zpq {

// The AES S-box (FIPS-197 figure 7), as an initializer list shared by the host key schedule and the device table build.
#define ZPQ_AES_SBOX                                                                                                    \
  {0x63, 0x7c, 0x77, 0x7b, 0xf2, 0x6b, 0x6f, 0xc5, 0x30, 0x01, 0x67, 0x2b, 0xfe, 0xd7, 0xab, 0x76, 0xca, 0x82, 0xc9,  \
   0x7d, 0xfa, 0x59, 0x47, 0xf0, 0xad, 0xd4, 0xa2, 0xaf, 0x9c, 0xa4, 0x72, 0xc0, 0xb7, 0xfd, 0x93, 0x26, 0x36, 0x3f,  \
   0xf7, 0xcc, 0x34, 0xa5, 0xe5, 0xf1, 0x71, 0xd8, 0x31, 0x15, 0x04, 0xc7, 0x23, 0xc3, 0x18, 0x96, 0x05, 0x9a, 0x07,  \
   0x12, 0x80, 0xe2, 0xeb, 0x27, 0xb2, 0x75, 0x09, 0x83, 0x2c, 0x1a, 0x1b, 0x6e, 0x5a, 0xa0, 0x52, 0x3b, 0xd6, 0xb3,  \
   0x29, 0xe3, 0x2f, 0x84, 0x53, 0xd1, 0x00, 0xed, 0x20, 0xfc, 0xb1, 0x5b, 0x6a, 0xcb, 0xbe, 0x39, 0x4a, 0x4c, 0x58,  \
   0xcf, 0xd0, 0xef, 0xaa, 0xfb, 0x43, 0x4d, 0x33, 0x85, 0x45, 0xf9, 0x02, 0x7f, 0x50, 0x3c, 0x9f, 0xa8, 0x51, 0xa3,  \
   0x40, 0x8f, 0x92, 0x9d, 0x38, 0xf5, 0xbc, 0xb6, 0xda, 0x21, 0x10, 0xff, 0xf3, 0xd2, 0xcd, 0x0c, 0x13, 0xec, 0x5f,  \
   0x97, 0x44, 0x17, 0xc4, 0xa7, 0x7e, 0x3d, 0x64, 0x5d, 0x19, 0x73, 0x60, 0x81, 0x4f, 0xdc, 0x22, 0x2a, 0x90, 0x88,  \
   0x46, 0xee, 0xb8, 0x14, 0xde, 0x5e, 0x0b, 0xdb, 0xe0, 0x32, 0x3a, 0x0a, 0x49, 0x06, 0x24, 0x5c, 0xc2, 0xd3, 0xac,  \
   0x62, 0x91, 0x95, 0xe4, 0x79, 0xe7, 0xc8, 0x37, 0x6d, 0x8d, 0xd5, 0x4e, 0xa9, 0x6c, 0x56, 0xf4, 0xea, 0x65, 0x7a,  \
   0xae, 0x08, 0xba, 0x78, 0x25, 0x2e, 0x1c, 0xa6, 0xb4, 0xc6, 0xe8, 0xdd, 0x74, 0x1f, 0x4b, 0xbd, 0x8b, 0x8a, 0x70,  \
   0x3e, 0xb5, 0x66, 0x48, 0x03, 0xf6, 0x0e, 0x61, 0x35, 0x57, 0xb9, 0x86, 0xc1, 0x1d, 0x9e, 0xe1, 0xf8, 0x98, 0x11,  \
   0x69, 0xd9, 0x8e, 0x94, 0x9b, 0x1e, 0x87, 0xe9, 0xce, 0x55, 0x28, 0xdf, 0x8c, 0xa1, 0x89, 0x0d, 0xbf, 0xe6, 0x42,  \
   0x68, 0x41, 0x99, 0x2d, 0x0f, 0xb0, 0x54, 0xbb, 0x16}

// An expanded AES encryption key: 4 * (rounds + 1) round-key words, big-endian (FIPS-197 5.2), rounds = 10 / 12 / 14.
struct AesKey {
  uint32_t rk[60];
  int rounds;
};
// keylen must be 16, 24 or 32 (the caller checks).
void aes_expand_key(const uint8_t* key, int keylen, AesKey& out);
// Overwrite memory that held key material so that the compiler cannot drop the stores.
void secure_zero(void* p, size_t n);

// One AES encryption of the block (s0, s1, s2, s3) (big-endian words) in place.  T(x) returns T0[x] =
// {02}S[x] << 24 | S[x] << 16 | S[x] << 8 | {03}S[x]; T1..T3 are its byte rotations, and the last round takes S[x] from
// bits 8..15 of T0[x], so one 256-word table is all the cipher reads.
template <int NR, class Tab>
__host__ __device__ __forceinline__ void aes_encrypt_words(const uint32_t* rk, const Tab& T, uint32_t& s0, uint32_t& s1,
                                                           uint32_t& s2, uint32_t& s3) {
#define ZPQ_ROR(x, k) (((x) >> (k)) | ((x) << (32 - (k))))
  s0 ^= rk[0]; s1 ^= rk[1]; s2 ^= rk[2]; s3 ^= rk[3];
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int r = 1; r < NR; ++r) {
    const uint32_t t0 = T(s0 >> 24) ^ ZPQ_ROR(T((s1 >> 16) & 255), 8) ^ ZPQ_ROR(T((s2 >> 8) & 255), 16) ^ ZPQ_ROR(T(s3 & 255), 24) ^ rk[4 * r];
    const uint32_t t1 = T(s1 >> 24) ^ ZPQ_ROR(T((s2 >> 16) & 255), 8) ^ ZPQ_ROR(T((s3 >> 8) & 255), 16) ^ ZPQ_ROR(T(s0 & 255), 24) ^ rk[4 * r + 1];
    const uint32_t t2 = T(s2 >> 24) ^ ZPQ_ROR(T((s3 >> 16) & 255), 8) ^ ZPQ_ROR(T((s0 >> 8) & 255), 16) ^ ZPQ_ROR(T(s1 & 255), 24) ^ rk[4 * r + 2];
    const uint32_t t3 = T(s3 >> 24) ^ ZPQ_ROR(T((s0 >> 16) & 255), 8) ^ ZPQ_ROR(T((s1 >> 8) & 255), 16) ^ ZPQ_ROR(T(s2 & 255), 24) ^ rk[4 * r + 3];
    s0 = t0; s1 = t1; s2 = t2; s3 = t3;
  }
#define ZPQ_SB(x) ((T(x) >> 8) & 255)
  const uint32_t* k = rk + 4 * NR;
  const uint32_t t0 = (ZPQ_SB(s0 >> 24) << 24 | ZPQ_SB((s1 >> 16) & 255) << 16 | ZPQ_SB((s2 >> 8) & 255) << 8 | ZPQ_SB(s3 & 255)) ^ k[0];
  const uint32_t t1 = (ZPQ_SB(s1 >> 24) << 24 | ZPQ_SB((s2 >> 16) & 255) << 16 | ZPQ_SB((s3 >> 8) & 255) << 8 | ZPQ_SB(s0 & 255)) ^ k[1];
  const uint32_t t2 = (ZPQ_SB(s2 >> 24) << 24 | ZPQ_SB((s3 >> 16) & 255) << 16 | ZPQ_SB((s0 >> 8) & 255) << 8 | ZPQ_SB(s1 & 255)) ^ k[2];
  const uint32_t t3 = (ZPQ_SB(s3 >> 24) << 24 | ZPQ_SB((s0 >> 16) & 255) << 16 | ZPQ_SB((s1 >> 8) & 255) << 8 | ZPQ_SB(s2 & 255)) ^ k[3];
  s0 = t0; s1 = t1; s2 = t2; s3 = t3;
#undef ZPQ_SB
#undef ZPQ_ROR
}

// libzpaq AES_CTR::encrypt(buf, n, offset) on a device buffer: buf[k] ^= keystream byte offset + k, keystream block j =
// AES_K(iv[0..7] || BE64(j)) (iv null = 8 zero bytes).  Asynchronous on `s`.
cudaError_t launch_aes_ctr(const AesKey& key, const uint8_t* iv8, uint8_t* d_buf, uint64_t n, uint64_t offset, cudaStream_t s);

// ---- host (zpq_crypto_host.cpp) ----
// scrypt per RFC 7914 (over PBKDF2-HMAC-SHA256).  Throws Failure(ZPQ_E_ARG) on bad parameters, Failure(ZPQ_E_NOMEM) when 128 * r * n bytes cannot be had.
void scrypt(const uint8_t* pw, uint64_t pwlen, const uint8_t* salt, uint64_t saltlen, uint64_t n, uint32_t r, uint32_t p,
            uint8_t* out, uint64_t outlen);

}  // namespace zpq
