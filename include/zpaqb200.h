/* zpaqb200.h -- C ABI of libzpaqb200.so, the B200-native ZPAQ block codec.
 *
 * This is the drop-in boundary for the compress / decompress hot path of mnadareski/ZPAQSharp
 * (a C# transliteration of libzpaq 7.12).  Every entry point names the reference interface it
 * replaces (file:line relative to /root/reference/ZPAQSharp).  The C# side keeps its LibZPAQ /
 * Compressor / Decompresser / Reader / Writer surface and calls these functions through
 * P/Invoke (see INTEGRATION.md for the binding stubs).
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every buffer; nothing is retained after return
 *   - "blocks" are ZPAQ archive blocks: independent units, one per resident warp on the device
 *   - block i of a batch occupies in[in_off[i] .. in_off[i+1]) ; offsets arrays have nb+1 entries
 *   - return value 0 = success, negative = error (ZPQ_E_*), message via zpq_last_error()
 *   - one zpq_ctx per host thread (not re-entrant); independent contexts are thread safe
 *   - all compute runs on the GPU(s) the context was created on; there is no CPU fallback:
 *     zpq_create fails when no CUDA device is usable
 */
#ifndef ZPAQB200_H
#define ZPAQB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zpq_ctx zpq_ctx;

enum {
  ZPQ_OK = 0,
  ZPQ_E_ARG = -1,        /* bad argument */
  ZPQ_E_CONFIG = -2,     /* method / config / header does not compile or is not supported */
  ZPQ_E_CUDA = -3,       /* CUDA runtime failure (message has the details) */
  ZPQ_E_NOMEM = -4,      /* device or host memory exhausted */
  ZPQ_E_OUTPUT = -5,     /* caller's output buffer too small (out_off[nb] holds the need if known) */
  ZPQ_E_CORRUPT = -6,    /* archive damaged (Decoder.cs:141, ZPAQL.cs:128-148, Decompresser.cs:49-53) */
  ZPQ_E_UNSUPPORTED = -7 /* valid input this build cannot process on the device */
};

/* Per-block status written by the kernels (zpq_block_status). */
enum {
  ZPQ_BLOCK_OK = 0,
  ZPQ_BLOCK_OVERFLOW = 1,   /* output slot too small */
  ZPQ_BLOCK_CORRUPT = 2,    /* "archive corrupted" / bad end of stream */
  ZPQ_BLOCK_ZPAQL = 3,      /* "ZPAQL execution error" */
  ZPQ_BLOCK_POSTPROC = 4    /* "unknown post processing type" / "Empty PCOMP" / unexpected EOS */
};

/* ---- context ----------------------------------------------------------------------------- */

/* Create a context bound to ndev CUDA devices (device_ids may be NULL = devices 0..ndev-1;
 * ndev <= 0 means "the current device only").  Replaces nothing in the reference (it has no
 * context object; Compressor/Decompresser instances own their state, Compressor.cs:15-18). */
int zpq_create(const int* device_ids, int ndev, zpq_ctx** out);
void zpq_destroy(zpq_ctx* ctx);

/* Message of the last failure on this context (or of the last failed zpq_create when ctx is
 * NULL).  Replaces LibZPAQ.error(string), LibZPAQ.cs:22-24: the C# wrapper forwards the text. */
const char* zpq_last_error(zpq_ctx* ctx);

/* Run the kernels of device 0 of this context on an existing CUDA stream (a cudaStream_t cast
 * to void*), e.g. the caller's current stream, so that the caller's events bracket the work.
 * NULL restores the context's own stream. */
int zpq_set_stream(zpq_ctx* ctx, void* cuda_stream);

/* Limit how many blocks are resident (being coded at once) per device; 0 = as many as fit. */
int zpq_set_max_resident(zpq_ctx* ctx, uint32_t max_blocks);

/* ---- model front end (host) ---------------------------------------------------------------- */

/* makeConfig(method, args), LibZPAQ.cs:388-1044: expand an "x.." / "s.." / "i.." / "0.." method
 * string into ZPAQL config text; args9 receives $1..$9.  Returns the text length (excluding the
 * NUL) or a negative error; text_cap may be 0 to query the length. */
int64_t zpq_make_config(const char* method, int* args9, char* text, uint64_t text_cap);

/* The digit-level expansion inside compressBlock, LibZPAQ.cs:128-283: "LB,R,t" plus the block's
 * bytes (level >= 5 analyses them) -> "x.." method string.  Returns its length or an error. */
int64_t zpq_expand_method(const char* method, const uint8_t* block, uint64_t n, char* out, uint64_t cap);

/* Compiler(config, args, hz, pz, pcomp_cmd), Compiler.cs:13-111.  hdr receives the block header
 * exactly as ZPAQL.write(out,false) emits it (ZPAQL.cs:158-179); pcomp receives the PCOMP
 * program including its END byte (length 0 if none). */
int zpq_compile_config(const char* config, const int* args9, uint8_t* hdr, uint64_t hdr_cap, uint64_t* hdr_len,
                       uint8_t* pcomp, uint64_t pcomp_cap, uint64_t* pcomp_len);

/* Header bytes of the built-in models of Compressor.startBlock(int level), Compressor.cs:45-83
 * (1 = min.cfg, 2 = mid.cfg, 3 = max.cfg).  Returns the length or an error. */
int64_t zpq_builtin_model(int level, uint8_t* hdr, uint64_t hdr_cap);

/* ZPAQL.memory(), ZPAQL.cs:58-81, for a header as stored in an archive.  Negative on error. */
double zpq_block_memory(const uint8_t* hdr, uint64_t hdr_len);

/* Bytes of device state one resident block of this model needs (tables + H/M/R), i.e. what the
 * scheduler divides free HBM by.  Negative on error. */
int64_t zpq_device_state_bytes(const uint8_t* hdr, uint64_t hdr_len, int for_decode);
/* The same when no block of the batch is longer than max_block_bytes: a MATCH component's history buffer (Predictor.cs:114-119,
 * ht of 2^bufbits bytes indexed by the stream position) is then allocated at the size the stream can reach, which holds the same
 * bytes at every index the component forms (mid.cfg with 1 MB blocks: 97 MB instead of 111 MB per block). */
int64_t zpq_device_state_bytes_for(const uint8_t* hdr, uint64_t hdr_len, int for_decode, uint64_t max_block_bytes);

/* How the role-split encoder (zpq_duo.cuh) would run this model with `smem_bytes` of shared memory per SM and
 * `blocks_per_sm` resident blocks wanted: the device analogue of asking the reference whether its x86 JIT applies
 * (Predictor.assemble_p, Predictor.cs:579-1356).  Host only, no device needed.  out[0..7] =
 *   [0] 1 if the role-split encoder applies, else 0 (the single-warp encoders are used)
 *   [1] lanes per block in a role warp (8, 16 or 32)          [2] role warps per block group (3 or 4)
 *   [3] blocks per SM that fit (<= blocks_per_sm)              [4] shared-memory bytes per resident block
 *   [5] coder delay in bits (Plan::coder_delay)                [6] 1 if the MIX components get a warp of their own
 *   [7] warps per CTA.                                          Returns 0 or a negative error code. */
int zpq_encoder_plan(const uint8_t* hdr, uint64_t hdr_len, uint32_t smem_bytes, uint32_t blocks_per_sm, int32_t* out8);

/* ---- compression --------------------------------------------------------------------------- */

/* LibZPAQ.compressBlock(in, out, method, filename, comment, dosha1), LibZPAQ.cs:117-325, for nb
 * independent blocks at once.  Each block becomes one complete archive block (13-byte tag,
 * header, one segment, trailer) written to out[out_off[i] .. out_off[i+1]); the concatenation is
 * what LibZPAQ.Compress (LibZPAQ.cs:84-108) writes for the same block split.  filename0 /
 * comment0 apply to the first block only (LibZPAQ.cs:104-105).  `method` is either a digit level
 * string ("2", "30,128,1") or an explicit "x.." string. */
int zpq_compress_blocks(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, const char* method,
                        const char* filename0, const char* comment0, int dosha1, uint8_t* out, uint64_t out_cap,
                        uint64_t* out_off);

/* Compressor.startBlock(int level) + startSegment + compress + endSegment + endBlock
 * (Compressor.cs:45-83,133-146,193-248,294-299) for nb blocks: built-in model `level`, one
 * segment per block, comment = decimal block size, SHA-1 trailer when dosha1, preceded by the
 * locator tag when with_tag (LibZPAQ.cs:296 writes it; a bare Compressor user may not). */
int zpq_compress_blocks_level(zpq_ctx* ctx, int level, const uint8_t* in, const uint64_t* in_off, uint32_t nb,
                              const char* filename0, const char* comment0, int dosha1, int with_tag, uint8_t* out,
                              uint64_t out_cap, uint64_t* out_off);

/* Compressor.startBlock(hcomp bytecode), Compressor.cs:85-99, plus an optional PCOMP program
 * (Compressor.postProcess, Compressor.cs:156-190) and the 9 method arguments that select the
 * pre-processing (args9[1], LibZPAQ.cs:301-312); otherwise as zpq_compress_blocks_level.  The
 * comment written is comment0 if given, else the decimal block size. */
int zpq_compress_blocks_model(zpq_ctx* ctx, const uint8_t* hdr, uint64_t hdr_len, const uint8_t* pcomp,
                              uint64_t pcomp_len, const int* args9, const uint8_t* in, const uint64_t* in_off,
                              uint32_t nb, const char* filename0, const char* comment0, int dosha1, int with_tag,
                              uint8_t* out, uint64_t out_cap, uint64_t* out_off);

/* Device-resident variant of zpq_compress_blocks_model used for kernel-only measurements: d_in,
 * d_in_off, d_out, d_out_off are DEVICE pointers on device 0 of the context; d_out receives the
 * same bytes, compacted; d_out_off[nb+1] is written on the device.  No host<->device copy of
 * block data happens inside.  Work is enqueued on the context's stream and completed (stream
 * synchronised) before return. */
int zpq_compress_blocks_model_dev(zpq_ctx* ctx, const uint8_t* hdr, uint64_t hdr_len, const uint8_t* pcomp,
                                  uint64_t pcomp_len, const int* args9, const uint8_t* d_in,
                                  const uint64_t* h_in_off, uint32_t nb, int dosha1, int with_tag, uint8_t* d_out,
                                  uint64_t out_cap, uint64_t* h_out_off);

/* ---- decompression ------------------------------------------------------------------------- */

/* Decompresser.findBlock, Decompresser.cs:29-58, over a whole archive in memory: reports the
 * byte offset of every block (position of its "zPQ") and of its end (one past the 255 byte).
 * offsets receives pairs (start,end); returns the number of blocks found or a negative error. */
int64_t zpq_find_blocks(const uint8_t* archive, uint64_t n, uint64_t* offsets, uint64_t max_blocks);

/* LibZPAQ.decompress(in, out), LibZPAQ.cs:65-79, for nb archive blocks at once: block i is
 * in[in_off[i] .. in_off[i+1]) and may start at its locator tag or at "zPQ".  All segments of a
 * block are decoded and concatenated into out[out_off[i] .. out_off[i+1]).  sha1_status (may be
 * NULL) receives per block: 0 = no segment stores a checksum, 1 = the SHA-1 of every segment that stores one matched the
 * restored bytes of that segment (hashed on the device), 2 = at least one did not
 * (Decompresser.readSegmentEnd, Decompresser.cs:163-194).  block_status (may be NULL) receives
 * ZPQ_BLOCK_* per block; a damaged block does not stop the batch, the call then returns
 * ZPQ_E_CORRUPT after decoding the others. */
int zpq_decompress_blocks(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, uint8_t* out,
                          uint64_t out_cap, uint64_t* out_off, uint8_t* sha1_status, uint8_t* block_status);

/* Upper bound of the decompressed size of the given blocks (from the decimal size compressBlock
 * stores in the segment comment, LibZPAQ.cs:298-300; blocks without one are estimated).  Lets
 * the caller size `out`. */
int64_t zpq_decompressed_bound(const uint8_t* in, const uint64_t* in_off, uint32_t nb);

/* ---- encryption ---------------------------------------------------------------------------- */

/* libzpaq 7.12's scrypt(pw, pwlen, salt, saltlen, n, r, p, out, outlen) (RFC 7914), which stretchKey calls
 * (StretchKey.cs:13-163 restates it).  Host only, no context.  n must be a power of two >= 2, r >= 1, p >= 1
 * (ZPQ_E_ARG otherwise); ZPQ_E_NOMEM when the 128 * r * n bytes of ROMix cannot be had.  outlen = 0 does nothing. */
int zpq_scrypt(const uint8_t* pw, uint64_t pwlen, const uint8_t* salt, uint64_t saltlen, uint64_t n, uint32_t r, uint32_t p,
               uint8_t* out, uint64_t outlen);

/* libzpaq stretchKey(out32, in32, salt32), StretchKey.cs:13-163: scrypt(in32, 32, salt32, 32, 16384, 8, 1, out32, 32).
 * As in libzpaq, in32 is SHA-256 of the password, computed by the caller.  Host only, no context. */
int zpq_stretch_key(const uint8_t* in32, const uint8_t* salt32, uint8_t* out32);

/* libzpaq AES_CTR(key, keylen, iv).encrypt(buf, n, offset) (the AES_CTR class of libzpaq 7.12; the reference has it as
 * prose only, LICENSE:635-665), on the device, in place on a HOST buffer: buf[k] ^= byte (offset + k) % 16 of
 * AES_key(iv[0..7] || big-endian 64-bit (offset + k) / 16).  iv8 may be NULL (8 zero bytes); keylen is 16, 24 or 32.
 * Encryption and decryption are the same call.  A context over N devices gives each a contiguous byte range; every device
 * works through at most 1 GiB of device memory at a time.  ZPQ_E_ARG for a bad key length, a NULL buffer with n > 0 or
 * offset + n past 2^64 - 1; n = 0 does nothing.  No key material is kept after return. */
int zpq_aes_ctr(zpq_ctx* ctx, const uint8_t* key, int keylen, const uint8_t* iv8, uint8_t* buf, uint64_t n, uint64_t offset);

/* The same on a DEVICE buffer of device 0 of the context (no host<->device copy): enqueued on that device's stream (the
 * context's own or the one zpq_set_stream gave) and completed before return, like zpq_compress_blocks_model_dev. */
int zpq_aes_ctr_dev(zpq_ctx* ctx, const uint8_t* key, int keylen, const uint8_t* iv8, uint8_t* d_buf, uint64_t n,
                    uint64_t offset);

/* ---- introspection ------------------------------------------------------------------------- */

/* Timing and launch statistics of the last compress / decompress / AES call on device 0.  For zpq_aes_ctr and
 * zpq_aes_ctr_dev: kernel_ms, h2d/d2h_ms and _bytes (host-buffer call; summed over its chunks), total_ms, launches, and
 * kernel = "aes_ctr/128", "aes_ctr/192" or "aes_ctr/256"; the other fields are 0. */
typedef struct zpq_stats {
  double h2d_ms, kernel_ms, d2h_ms, total_ms; /* CUDA-event times on the context's stream */
  double codec_kernel_ms;                      /* the coding kernel alone */
  uint64_t h2d_bytes, d2h_bytes;
  uint32_t launches;                           /* kernels launched */
  uint32_t resident_blocks;                    /* blocks coded concurrently */
  uint64_t state_bytes_per_block;
  char kernel[96];                             /* which coding kernel ran: "lanes/aot2 (HCOMP compiled)", "lanes/nvrtc", ... */
  double post_kernel_ms;                       /* decode: the post-processing pass (PostProcessor.cs:37-86) behind the decoding kernel */
  uint32_t post_native_blocks;                 /* decode: blocks restored by a native kernel (PASS copy, LZ77, BWT, E8E9) ... */
  uint32_t post_interpreted_blocks;            /* ... blocks whose stored PCOMP program was interpreted ... */
  uint32_t post_compiled_blocks;               /* ... and blocks whose stored program ran as NVRTC-compiled code */
  uint32_t reserved0;
} zpq_stats;
int zpq_get_stats(zpq_ctx* ctx, zpq_stats* out);

/* Model specialisation, the device analogue of the reference's x86 JIT (ZPAQL.assemble,
 * ZPAQL.cs:353-1008; Predictor.assemble_p, Predictor.cs:579-1356): generate the CUDA source of the
 * lane-resident kernels for this header and compile it with NVRTC for sm_100a.  Needs no GPU.
 * Returns the cubin size, or a negative error with the compiler log in `log`; `source` (may be
 * NULL) receives the generated text. */
int64_t zpq_specialize_model(const uint8_t* hdr, uint64_t hdr_len, char* source, uint64_t source_cap, char* log,
                             uint64_t log_cap);

/* Which post-processor the decoder uses for a block whose header says (ph, pm) and whose first segment stores the PCOMP
 * program pcomp[0..len): 0 = the stored program is interpreted (PostProcessor.write + ZPAQL.run, PostProcessor.cs:37-86);
 * otherwise kind | e8 << 4 | param << 8 with kind 2 = "lazy2" bit-packed LZ77 (LibZPAQ.cs:430-571; param = rb), 3 = "lzpre"
 * byte-aligned LZ77 (:577-638; param = minMatch), 4 = "bwtrle" inverse BWT (:644-794), 5 = "e8e9" (:801-826); e8 = the
 * program ends with the inverse E8E9 pass.  The programs are recognised byte for byte against what makeConfig emits. */
int64_t zpq_post_kind(int ph, int pm, const uint8_t* pcomp, uint64_t len);

/* The device analogue of the reference's x86 JIT for PCOMP (ZPAQL.assemble, ZPAQL.cs:353-1008): translate a PCOMP program to
 * CUDA and compile it with NVRTC for sm_100a, as the decoder does for stored programs that are not one of makeConfig's four
 * (ZPQ_POST_NVRTC=0 leaves them to the interpreter).  Needs no GPU.  Returns the cubin size, or a negative error with the
 * compiler log in `log`; `source` (may be NULL) receives the generated text. */
int64_t zpq_specialize_pcomp(int ph, int pm, const uint8_t* pcomp, uint64_t len, char* source, uint64_t source_cap, char* log,
                             uint64_t log_cap);

/* Library / build identification: "zpaqb200 <version> sm_100a". */
const char* zpq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ZPAQB200_H */
