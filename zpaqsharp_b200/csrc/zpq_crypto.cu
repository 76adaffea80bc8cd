// zpq_crypto.cu -- libzpaq 7.12's AES_CTR::encrypt(buf, n, offset) on the device (zpaq's -key archives).
//
// Byte offset + k of the stream is XORed with byte (offset + k) % 16 of keystream block j = (offset + k) / 16, and keystream
// block j is AES_K(iv[0..7] || BE64(j)).  Every keystream block is independent, so the kernel is a grid-stride loop over them.
//
// Round function: one 256-word T-table in shared memory, T1..T3 as byte rotations of it, the last round's S-box byte taken
// out of T0 (see aes_encrypt_words).  The table is replicated 32 times, laid out [256][32], and lane l reads only column l:
// word x * 32 + l sits in bank l whatever x is, so no look-up ever conflicts and the shared-memory timing of a warp does not
// depend on the key or the counter.
#include <cuda_runtime.h>
#include <stdint.h>

#include "zpq_crypto.h"

namespace zpq {

namespace {

constexpr int kThreads = 256;   // 8 warps per CTA; the 32 KB table is shared by all of them
constexpr int kPer = 4;         // keystream blocks per thread per pass: a warp covers 128 consecutive blocks, lane l blocks l, l+32, ..

__constant__ uint8_t c_sbox[256] = ZPQ_AES_SBOX;

struct AesCtrParams {
  uint32_t rk[60];
  uint32_t iv0, iv1;            // iv as big-endian words
  uint8_t* buf;
  uint64_t n;
  uint64_t jfirst;              // keystream block of buf[0]
  uint64_t m;                   // keystream blocks that touch buf
  uint32_t r;                   // offset % 16
  uint32_t wide;                // alignment of the whole blocks inside buf: 16, 4 or 1 bytes
};

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// XOR keystream block i of this call (words ks, big-endian) into the bytes of buf it covers.
__device__ __forceinline__ void apply_block(const AesCtrParams& p, uint64_t i, const uint32_t (&ks)[4]) {
  const uint64_t lo = 16 * i - p.r;                       // buffer index of the block's byte 0 (wraps for i = 0, r > 0)
  const bool whole = (i > 0 || p.r == 0) && lo + 16 <= p.n;
  if (whole && p.wide == 16) {
    uint4* q = reinterpret_cast<uint4*>(p.buf + lo);
    uint4 v = *q;
    v.x ^= bswap32(ks[0]); v.y ^= bswap32(ks[1]); v.z ^= bswap32(ks[2]); v.w ^= bswap32(ks[3]);
    *q = v;
  } else if (whole && p.wide == 4) {
    uint32_t* q = reinterpret_cast<uint32_t*>(p.buf + lo);
#pragma unroll
    for (int t = 0; t < 4; ++t) q[t] ^= bswap32(ks[t]);
  } else {                                                // head, tail, or a buffer aligned to less than 4 bytes
#pragma unroll
    for (int b = 0; b < 16; ++b) {
      const uint64_t at = lo + b;
      if ((i > 0 || (uint32_t)b >= p.r) && at < p.n) p.buf[at] ^= (uint8_t)(ks[b >> 2] >> (24 - 8 * (b & 3)));
    }
  }
}

template <int NR>
__global__ void __launch_bounds__(kThreads) k_aes_ctr(const __grid_constant__ AesCtrParams p) {
  __shared__ uint32_t tab[256 * 32];
  for (int e = threadIdx.x; e < 256 * 32; e += kThreads) {
    const uint32_t s = c_sbox[e >> 5];
    const uint32_t s2 = ((s << 1) ^ ((s >> 7) * 0x11b)) & 255;   // {02} * s in GF(2^8)
    tab[e] = s2 << 24 | s << 16 | s << 8 | (s2 ^ s);
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t* col = tab + lane;
  const auto T = [col](uint32_t x) { return col[x << 5]; };
  const uint64_t span = 32 * kPer;
  const uint64_t step = (uint64_t)gridDim.x * (kThreads / 32) * span;
  for (uint64_t base = ((uint64_t)blockIdx.x * (kThreads / 32) + threadIdx.x / 32) * span; base < p.m; base += step) {
    uint32_t ks[kPer][4];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const uint64_t j = p.jfirst + base + k * 32 + lane;
      ks[k][0] = p.iv0; ks[k][1] = p.iv1; ks[k][2] = (uint32_t)(j >> 32); ks[k][3] = (uint32_t)j;
      aes_encrypt_words<NR>(p.rk, T, ks[k][0], ks[k][1], ks[k][2], ks[k][3]);
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const uint64_t i = base + k * 32 + lane;
      if (i < p.m) apply_block(p, i, ks[k]);
    }
  }
}

template <int NR>
cudaError_t launch_nr(const AesCtrParams& p, cudaStream_t s) {
  int dev = 0, sms = 0, per_sm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_aes_ctr<NR>, kThreads, 0);
  if (e != cudaSuccess) return e;
  const uint64_t per_cta = (uint64_t)(kThreads / 32) * 32 * kPer;
  const uint64_t want = (p.m + per_cta - 1) / per_cta;
  const uint64_t wave = (uint64_t)sms * (uint64_t)(per_sm > 0 ? per_sm : 1);
  const unsigned grid = (unsigned)(want < wave ? want : wave);
  k_aes_ctr<NR><<<grid, kThreads, 0, s>>>(p);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_aes_ctr(const AesKey& key, const uint8_t* iv8, uint8_t* d_buf, uint64_t n, uint64_t offset, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  AesCtrParams p;
  for (int i = 0; i < 60; ++i) p.rk[i] = i < 4 * (key.rounds + 1) ? key.rk[i] : 0;
  p.iv0 = iv8 ? (uint32_t)iv8[0] << 24 | (uint32_t)iv8[1] << 16 | (uint32_t)iv8[2] << 8 | iv8[3] : 0;
  p.iv1 = iv8 ? (uint32_t)iv8[4] << 24 | (uint32_t)iv8[5] << 16 | (uint32_t)iv8[6] << 8 | iv8[7] : 0;
  p.buf = d_buf;
  p.n = n;
  p.jfirst = offset / 16;
  p.m = (offset + n - 1) / 16 - offset / 16 + 1;
  p.r = (uint32_t)(offset % 16);
  const uintptr_t first_whole = (uintptr_t)d_buf - p.r;   // where block 1 starts, minus 16
  p.wide = first_whole % 16 == 0 ? 16 : first_whole % 4 == 0 ? 4 : 1;
  cudaError_t e = key.rounds == 10 ? launch_nr<10>(p, s) : key.rounds == 12 ? launch_nr<12>(p, s) : launch_nr<14>(p, s);
  secure_zero(p.rk, sizeof p.rk);
  return e;
}

}  // namespace zpq
