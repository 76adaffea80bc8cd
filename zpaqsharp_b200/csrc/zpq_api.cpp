// zpq_api.cpp -- C ABI of libzpaqb200 and the host scheduler behind it.
//
// The scheduler turns a batch of independent archive blocks into device work:
//   compress:   H2D -> [SHA-1] -> [E8E9] -> encode kernel (one warp per resident block, atomic
//               block queue) -> frame assembly -> scan -> gather -> D2H
//   decompress: host parses block/segment framing (a few hundred bytes per block), H2D ->
//               decode kernel (+ ZPAQL post-processing on the device) -> [SHA-1] -> scan ->
//               gather -> D2H
// Blocks never communicate, so multi-GPU use is a plain partition of the block list; results are
// concatenated in block order (no collective).
//
// There is no CPU fallback: every entry point that touches block data fails when CUDA fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <condition_variable>
#include <map>
#include <memory>
#include <mutex>
#include <atomic>
#include <thread>

#include "zpq_aot.h"
#include "zpq_crypto.h"
#include "zpq_device.h"
#include "zpq_host.h"

namespace zpq {
bool find_spec_kernels(const Header& hdr, uint32_t smem_limit, SpecKernels& out, std::string* why_not);
void spec_set_smem_limit(uint32_t bytes);
Bytes nvrtc_compile(const std::string& src);
const void* find_post_kernel(const Bytes& prog, int ph, int pm, std::string* why_not);
int64_t post_program_cubin(const Bytes& prog, int ph, int pm, std::string* source, std::string* log);
std::string generate_model_source(const Header& hdr, const std::string& name, const std::string& enc_kernel,
                                  const std::string& dec_kernel, bool* compiled_hcomp, int* duo_g, bool* fdec);
}

using namespace zpq;

namespace {

#define CU(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      throw Failure(e__ == cudaErrorMemoryAllocation ? ZPQ_E_NOMEM : ZPQ_E_CUDA,                   \
                    std::string(#expr) + ": " + cudaGetErrorString(e__));                          \
  } while (0)

std::string g_create_error;
std::mutex g_create_mutex;

inline uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

// Grow-only device buffer.
struct DevBuf {
  void* p = nullptr;
  uint64_t cap = 0;
  void reserve(uint64_t bytes) {
    if (bytes <= cap) return;
    release();
    CU(cudaMalloc(&p, bytes));
    cap = bytes;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
  }
  template <class T> T* as() const { return static_cast<T*>(p); }
};

// Reserve an I/O buffer; if the device is full because an earlier call's state arenas still hold
// the memory, drop them and try again.
void reserve_io(DevBuf& b, uint64_t bytes, DevBuf& arena) {
  try { b.reserve(bytes); }
  catch (const Failure& f) {
    if (f.code != ZPQ_E_NOMEM || !arena.p) throw;
    cudaGetLastError();
    arena.release();
    b.reserve(bytes);
  }
}

struct Timer {
  cudaEvent_t a = nullptr, b = nullptr;
  void init() { CU(cudaEventCreate(&a)); CU(cudaEventCreate(&b)); }
  void fini() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); a = b = nullptr; }
  void start(cudaStream_t s) { CU(cudaEventRecord(a, s)); }
  void stop(cudaStream_t s) { CU(cudaEventRecord(b, s)); }
  double ms() const { float t = 0; cudaEventElapsedTime(&t, a, b); return t; }
};

// What one group (one model header) of a decode batch owns while it runs: groups of different models run side by side, each on
// its own stream with its own raw-stream buffer, job tables, plan and state arenas.
struct Scratch {
  DevBuf work, meta, plan, arena;
  cudaStream_t stream = nullptr;
  Timer t_codec, t_post;
  void init() { CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); t_codec.init(); t_post.init(); }
  void release() { work.release(); meta.release(); plan.release(); arena.release(); }
  void fini() { release(); t_codec.fini(); t_post.fini(); if (stream) cudaStreamDestroy(stream); stream = nullptr; }
};
// Every group of a multi-model batch takes its memory before any of them launches: cudaMalloc / cudaFree wait for running kernels,
// so an allocation behind a launch would put the groups back in a row.
struct GroupBarrier {
  std::mutex m; std::condition_variable cv; size_t need = 0, got = 0;
  void arrive() { std::lock_guard<std::mutex> lk(m); ++got; cv.notify_all(); }
  void arrive_and_wait() { std::unique_lock<std::mutex> lk(m); ++got; cv.notify_all(); cv.wait(lk, [&] { return got >= need; }); }
};
struct GroupBufs { DevBuf& work; DevBuf& meta; DevBuf& plan; DevBuf& arena; cudaStream_t stream; Timer& t_codec; Timer& t_post; };

struct Device {
  int id = 0;
  cudaStream_t own = nullptr, stream = nullptr;
  std::vector<std::unique_ptr<Scratch>> pool;      // for the second, third ... group of a decode batch
  cudaEvent_t ev_ready = nullptr;
  int sms = 0;
  uint32_t smem_optin = 0;
  Tables* d_tab = nullptr;
  DevBuf arena, in, work, pre, slots, out, meta, plan;
  Timer t_all, t_h2d, t_kern, t_codec, t_d2h, t_post;
  zpq_stats stats{};

  void init(int dev) {
    id = dev;
    CU(cudaSetDevice(id));
    CU(cudaStreamCreateWithFlags(&own, cudaStreamNonBlocking));
    stream = own;
    int v = 0;
    CU(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, id)); sms = v;
    CU(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, id)); smem_optin = (uint32_t)v;
    CU(codec_set_smem_limit(smem_optin));
    spec_set_smem_limit(smem_optin);
    std::unique_ptr<Tables> t(new Tables);
    build_tables(*t);
    CU(cudaMalloc(&d_tab, sizeof(Tables)));
    CU(cudaMemcpy(d_tab, t.get(), sizeof(Tables), cudaMemcpyHostToDevice));
    t_all.init(); t_h2d.init(); t_kern.init(); t_codec.init(); t_d2h.init(); t_post.init();
    CU(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
  }
  void fini() {
    cudaSetDevice(id);
    arena.release(); in.release(); work.release(); pre.release(); slots.release(); out.release(); meta.release(); plan.release();
    if (d_tab) cudaFree(d_tab);
    for (auto& sc : pool) sc->fini();
    pool.clear();
    if (ev_ready) cudaEventDestroy(ev_ready);
    t_all.fini(); t_h2d.fini(); t_kern.fini(); t_codec.fini(); t_d2h.fini(); t_post.fini();
    if (own) cudaStreamDestroy(own);
  }
};

// A model as the codec needs it.
struct Model {
  Header hdr;
  Bytes pcomp;     // program incl. END, may be empty
  int args[9];
};

// Geometry of a codec launch for `want` blocks of this model.
struct Launch {
  std::unique_ptr<Plan> plan;
  SmemLayout sm;
  LaunchGeom geom;
  uint32_t resident;
  SpecKernels spec;        // specialised kernels for this header, if any
  bool has_spec = false;
  bool skewed = false;     // encode with the time-skewed kernel (zpq_pipe.cuh)
  bool duo = false;        // encode with the two-role kernel (zpq_duo.cuh)
  bool fast = false;       // decode with the speculative kernel (zpq_fdec.cuh); the post-processor is a separate pass
  uint32_t wb = 0;         // ... blocks per CTA
  uint32_t duo_roles = 3;  // ... role warps per block group (context, history, coder[, mixer])
  std::string kernel;      // what will run (for zpq_stats)
};

cudaError_t launch_codec(const Launch& L, const CodecParams& p, bool decode, cudaStream_t s) {
  if (L.has_spec) {
    void* args[] = {const_cast<CodecParams*>(&p)};
    const void* k = decode ? (L.fast ? L.spec.dec_fast : L.spec.dec) : L.duo ? L.spec.enc_duo : (L.skewed ? L.spec.enc : L.spec.enc_lanes);
    // the dynamic shared memory limit is a per-device attribute (NVRTC kernels are shared by all devices of the process)
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.sm.total);
    if (e != cudaSuccess) return e;
    return cudaLaunchKernel(k, dim3(L.geom.grid), dim3(L.geom.warps_per_cta * 32), args, p.sm.total, s);
  }
  return decode ? launch_decode(p, L.geom, s) : launch_encode(p, L.geom, s);
}

uint32_t common_smem(const Plan& pl, SmemLayout& L) {
  uint32_t o = 0;
  bool with_dt = false;   // dt is only read by train() of CM and SSE components (Predictor.cs:1031-1036)
  for (int i = 0; i < pl.n; ++i) with_dt = with_dt || pl.comp[i].type == C_CM || pl.comp[i].type == C_SSE;
  L.stretch = 0; L.squash = 65536; L.dt2k = 73728; L.ns = 74240; L.dt = 75264;
  L.tables_bytes = with_dt ? 79360u : 75264u;
  o = L.tables_bytes;
  L.comp = o; o += (uint32_t)align_up((uint64_t)std::max(pl.n, 1) * sizeof(CompDesc), 16);
  L.order = o; o += (uint32_t)align_up(std::max(pl.n, 1), 16);
  L.steps = o; o += (uint32_t)align_up((uint64_t)std::max(pl.nsteps, 1) * sizeof(Step), 16);
  L.mix = o; o += (uint32_t)align_up((uint64_t)std::max(pl.nmix, 1) * sizeof(MixDesc), 16);
  if (pl.hcomp_len + 8 <= 4096) { L.hcomp = o; o += (uint32_t)align_up(pl.hcomp_len + 8, 16); }
  else L.hcomp = kNoSmem;
  return (uint32_t)align_up(o, 128);
}

bool force_generic();

void plan_launch(Device& d, const Header& hdr, bool decode, uint64_t want, uint64_t mem_for_arenas, uint32_t max_resident,
                 Launch& L, bool want_skew = false, bool want_duo = false, bool want_fast = false, uint64_t max_stream = 0) {
  L.plan.reset(new Plan);
  build_plan(hdr, decode, 48 * 1024, *L.plan, 0, false, max_stream);
  L.skewed = false; L.duo = false; L.wb = 0; L.fast = false;
  uint64_t fit = mem_for_arenas / std::max<uint64_t>(L.plan->arena_bytes, 1);
  if (fit < 1) throw Failure(ZPQ_E_NOMEM, "model state does not fit in device memory");
  uint64_t resident = std::min<uint64_t>({want, fit, (uint64_t)d.sms * 16});
  if (max_resident) resident = std::min<uint64_t>(resident, max_resident);
  if (resident < 1) resident = 1;
  uint32_t W = (uint32_t)((resident + d.sms - 1) / d.sms);
  W = std::max(1u, std::min(16u, W));
  SpecKernels spec;
  std::string why;
  const bool lanes = L.plan->lane_ok && !force_generic();
  const bool has_spec = lanes && find_spec_kernels(hdr, d.smem_optin, spec, &why);
  if (want_duo && has_spec && spec.enc_duo && !decode) {
    // Two-role encoder (zpq_duo.cuh): 32/G blocks share a pair of warps, up to 7 pairs per SM plus one
    // arithmetic coder warp (lane = block, so at most 32 blocks); every ICM/ISSE map has to live in the block's shared slice.
    const uint32_t G = (uint32_t)spec.duo_g, B = 32 / G;
    {
      std::unique_ptr<Plan> probe(new Plan);
      build_plan(hdr, false, 48 * 1024, *probe, (int)G, false, max_stream);
      L.duo_roles = probe->duo_split ? 4 : 3;
    }
    const uint32_t max_groups = 15u / L.duo_roles;     // 16 warps per CTA, one of them the arithmetic coder
    uint64_t res = std::min<uint64_t>({want, fit, (uint64_t)d.sms * std::min(max_groups * B, 32u)});
    if (max_resident) res = std::min<uint64_t>(res, max_resident);
    if (res < 1) res = 1;
    uint32_t wb = (uint32_t)((res + d.sms - 1) / d.sms);
    for (uint32_t w = wb; w >= 1 && !L.duo; --w) {
      const uint32_t common = common_smem(*L.plan, L.sm);
      const uint32_t avail = d.smem_optin > common ? d.smem_optin - common : 0;
      build_plan(hdr, false, (avail / w) & ~127u, *L.plan, (int)G, false, max_stream);
      if (L.plan->duo_ok && L.plan->pipe_maps && (uint64_t)w * L.plan->smem_warp_bytes <= avail) { L.duo = true; wb = w; }
    }
    if (L.duo) {
      res = std::min<uint64_t>(res, (uint64_t)wb * d.sms);
      L.sm.slices = common_smem(*L.plan, L.sm);
      L.sm.slice_bytes = L.plan->smem_warp_bytes;
      L.sm.total = L.sm.slices + wb * L.sm.slice_bytes;
      L.wb = wb;
      L.geom.warps_per_cta = 1 + L.duo_roles * ((wb + B - 1) / B);
      L.geom.lanes = 1;
      L.has_spec = true; L.spec = spec;
      L.kernel = std::string("duo/") + spec.origin + ", " + std::to_string(L.duo_roles) + " roles + coder warp, x" + std::to_string(B) + " blocks per warp";
      L.geom.grid = (uint32_t)((res + wb - 1) / wb);
      L.resident = (uint32_t)res;
      return;
    }
    build_plan(hdr, decode, 48 * 1024, *L.plan, 0, false, max_stream);
  }
  if (want_fast && has_spec && spec.dec_fast && decode) {
    // Speculative decoder (zpq_fdec.cuh): one warp per block, every ICM/ISSE map in the block's shared slice
    for (uint32_t w = std::min(W, 12u); w >= 1 && !L.fast; --w) {      // kFdecThreads = 384
      const uint32_t common = common_smem(*L.plan, L.sm);
      const uint32_t avail = d.smem_optin > common ? d.smem_optin - common : 0;
      build_plan(hdr, true, (avail / w) & ~127u, *L.plan, 0, true, max_stream);
      const bool hm_ok = ((4ull << hdr.hh) > 2048 || L.plan->smem_h != kNoSmem) && ((1ull << hdr.hm) > 1024 || L.plan->smem_m != kNoSmem);
      if (L.plan->pipe_maps && hm_ok && (uint64_t)w * L.plan->smem_warp_bytes <= avail) { L.fast = true; W = w; }
    }
    if (L.fast) {
      resident = std::min<uint64_t>(resident, (uint64_t)W * d.sms);
      L.sm.slices = common_smem(*L.plan, L.sm);
      L.sm.slice_bytes = L.plan->smem_warp_bytes;
      L.sm.total = L.sm.slices + W * L.sm.slice_bytes;
      L.geom.warps_per_cta = W;
      L.geom.lanes = 1;
      L.has_spec = true; L.spec = spec;
      L.kernel = std::string("fdec/") + spec.origin + ", speculative, post-processor as a second pass";
      L.geom.grid = (uint32_t)((resident + W - 1) / W);
      L.resident = (uint32_t)resident;
      return;
    }
    build_plan(hdr, decode, 48 * 1024, *L.plan, 0, false, max_stream);
  }
  if (want_skew && has_spec && !decode) {
    // The time-skewed encoder (zpq_pipe.cuh) keeps every ICM/ISSE map in the block's shared slice:
    // take the largest number of blocks per SM for which that holds.
    for (uint32_t w = W; w >= 1 && !L.skewed; --w) {
      const uint32_t common = common_smem(*L.plan, L.sm);
      const uint32_t avail = d.smem_optin > common ? d.smem_optin - common : 0;
      build_plan(hdr, decode, (avail / w) & ~127u, *L.plan, 0, false, max_stream);
      if (L.plan->pipe_ok && L.plan->pipe_maps && (uint64_t)w * L.plan->smem_warp_bytes <= avail) { L.skewed = true; W = w; }
    }
    if (!L.skewed) build_plan(hdr, decode, 48 * 1024, *L.plan, 0, false, max_stream);
  }
  for (;;) {
    uint32_t common = common_smem(*L.plan, L.sm);
    uint32_t avail = d.smem_optin > common ? d.smem_optin - common : 0;
    if ((uint64_t)W * L.plan->smem_warp_bytes <= avail) break;
    uint32_t budget = avail / W;
    uint32_t minimal = (uint32_t)align_up(24ull * std::max(hdr.n, 1) + 64 + 1024 + 256, 128) + (hdr.n <= 32 ? 4096u : 0u);
    if (budget >= minimal) {
      build_plan(hdr, decode, budget & ~127u, *L.plan, 0, false, max_stream);
      common = common_smem(*L.plan, L.sm);
      avail = d.smem_optin > common ? d.smem_optin - common : 0;
      if ((uint64_t)W * L.plan->smem_warp_bytes <= avail) break;
    }
    if (W == 1) throw Failure(ZPQ_E_UNSUPPORTED, "model needs more shared memory than one SM has");
    --W;
  }
  resident = std::min<uint64_t>(resident, (uint64_t)W * d.sms);
  L.sm.slices = common_smem(*L.plan, L.sm);
  L.sm.slice_bytes = L.plan->smem_warp_bytes;
  L.sm.total = L.sm.slices + W * L.sm.slice_bytes;
  L.geom.warps_per_cta = W;
  L.geom.lanes = lanes ? 1u : 0u;
  L.has_spec = has_spec;
  L.spec = spec;
  L.kernel = L.geom.lanes ? "lanes/generic" : "steps/generic";
  if (has_spec) L.kernel = std::string("lanes/") + spec.origin + (L.skewed ? ", time-skewed" : "");
  else if (lanes) L.kernel += " (" + why.substr(0, 60) + ")";
  L.geom.grid = (uint32_t)((resident + W - 1) / W);
  L.resident = (uint32_t)resident;
}

// ZPQ_FORCE_GENERIC=1 selects the step-scheduled kernels even for small models (test hook).
bool force_generic() { const char* e = getenv("ZPQ_FORCE_GENERIC"); return e && *e == '1'; }

uint64_t free_device_memory() {
  size_t fr = 0, tot = 0;
  CU(cudaMemGetInfo(&fr, &tot));
  return fr;
}

}  // namespace

struct zpq_ctx {
  std::vector<Device> devs;
  std::string err;
  uint32_t max_resident = 0;
};

namespace {

// ------------------------------------------------------------------------------------------
// Compression of blocks [first, first+count) of one model on one device.
// Input either on the host (h_in) or already on the device (d_in_ext).  Output frames are
// gathered into d_out (device) and, for host calls, copied to h_out + h_out_base.
// Returns total frame bytes; frame_off[0..count] (relative) is filled.
// ------------------------------------------------------------------------------------------
struct CompressTask {
  const Model* model;
  const uint8_t* h_in = nullptr;        // host input base (offsets are absolute into it)
  const uint8_t* d_in_ext = nullptr;    // or device input base
  const uint64_t* in_off = nullptr;     // host array, absolute offsets, nb+1 entries overall
  uint32_t first = 0, count = 0;
  std::vector<std::string> filenames, comments;  // per block of this task (may be empty strings)
  bool dosha1 = true, with_tag = true;
  uint8_t* d_out_ext = nullptr;         // device output (dev variant) or null
  uint64_t d_out_cap = 0;
  std::vector<uint64_t> frame_off;      // out: count+1
};

void build_prefix(const Model& m, const std::string& filename, const std::string& comment, bool with_tag, Bytes& out) {
  if (with_tag) out.insert(out.end(), kLocatorTag, kLocatorTag + 13);          // Compressor.cs:27-43
  out.push_back('z'); out.push_back('P'); out.push_back('Q');                  // Compressor.cs:109-113
  out.push_back((uint8_t)(1 + (m.hdr.n == 0)));
  out.push_back(1);
  out.insert(out.end(), m.hdr.wire.begin(), m.hdr.wire.end());                 // ZPAQL.write, ZPAQL.cs:158-179
  out.push_back(1);                                                            // Compressor.cs:133-146
  out.insert(out.end(), filename.begin(), filename.end()); out.push_back(0);
  out.insert(out.end(), comment.begin(), comment.end()); out.push_back(0);
  out.push_back(0);
}

uint64_t compress_on_device(zpq_ctx* ctx, Device& d, CompressTask& T, uint8_t* h_out, uint64_t h_out_cap) {
  CU(cudaSetDevice(d.id));
  cudaStream_t s = d.stream;
  const Model& M = *T.model;
  const uint32_t nb = T.count;
  const uint64_t* off = T.in_off + T.first;
  const uint64_t in_base = off[0], in_total = off[nb] - off[0];
  d.stats = zpq_stats{};
  d.t_all.start(s);

  const int pre = M.args[1];
  if (pre < 0 || pre > 7) throw Failure(ZPQ_E_CONFIG, "Unsupported method");
  const int lz_level = pre & 3;                       // 0 none, 1 bit-packed LZ77, 2 byte LZ77, 3 BWT   (LibZPAQ.cs:301-312)
  const bool do_e8 = pre >= 4;
  const bool use_sa = lz_level == 3 || (lz_level && M.args[5] - M.args[0] >= 21);
  if (lz_level == 1 && M.args[2] < 4) throw Failure(ZPQ_E_CONFIG, "match length $3 too small");
  if (lz_level == 2 && M.args[2] < 1) throw Failure(ZPQ_E_CONFIG, "match length $3 too small");
  if (lz_level && lz_level < 3 && !use_sa && (M.args[5] < 1 || M.args[5] > 28)) throw Failure(ZPQ_E_UNSUPPORTED, "LZ77 hash table size out of range");

  // ---- host-side metadata: preamble, prefixes, jobs ----
  Bytes preamble;
  if (!M.pcomp.empty()) {                                                      // Compressor.cs:177-188
    preamble.push_back(1);
    preamble.push_back((uint8_t)(M.pcomp.size() & 255));
    preamble.push_back((uint8_t)(M.pcomp.size() >> 8));
    preamble.insert(preamble.end(), M.pcomp.begin(), M.pcomp.end());
  } else preamble.push_back(0);

  Bytes prefix;
  std::vector<uint32_t> prefix_off(nb + 1);
  std::vector<EncJob> jobs(nb);
  std::vector<uint64_t> slot_off(nb + 1), rel_off(nb + 1), pre_off(nb + 1);
  uint64_t pre_total = 0, max_block = 0;
  std::vector<uint32_t> lens(nb);
  uint64_t slots_total = 0, max_frame = 0;
  for (uint32_t i = 0; i < nb; ++i) {
    const uint64_t n = off[i + 1] - off[i];
    if (n > 0xFFFFFFFFull - 8192) throw Failure(ZPQ_E_ARG, "block larger than 4 GiB");
    prefix_off[i] = (uint32_t)prefix.size();
    const std::string& cm = T.comments.size() > i && !T.comments[i].empty() ? T.comments[i] : std::to_string(n);
    build_prefix(M, T.filenames.size() > i ? T.filenames[i] : std::string(), cm, T.with_tag, prefix);
    const uint32_t plen = (uint32_t)prefix.size() - prefix_off[i];
    const uint64_t tlen = lz_level == 3 ? n + 5 : lz_level ? n + n / 16 + 64 : n;      // bound of the transformed stream
    pre_off[i] = pre_total; pre_total = align_up(pre_total + tlen + 16, 16);
    const uint64_t stream = tlen + preamble.size();
    const uint64_t cap = M.hdr.n ? stream + stream / 4 + 4096 : stream + 4 * (stream / 65536 + 1) + 16;
    slot_off[i] = slots_total;
    jobs[i].in_off = lz_level ? pre_off[i] : off[i] - in_base;
    jobs[i].in_len = lz_level ? 0u : (uint32_t)n;         // filled by the pre-processing kernels
    max_block = std::max(max_block, n);
    jobs[i].pre_len = (uint32_t)preamble.size();
    jobs[i].out_off = slots_total + plen;
    jobs[i].out_cap = cap;
    rel_off[i] = off[i] - in_base;
    lens[i] = (uint32_t)n;
    const uint64_t frame = plen + cap + 32;
    max_frame = std::max(max_frame, frame);
    slots_total = align_up(slots_total + frame, 16);
  }
  prefix_off[nb] = (uint32_t)prefix.size();
  slot_off[nb] = slots_total;
  rel_off[nb] = in_total;
  pre_off[nb] = pre_total;

  // ---- device buffers ----
  // meta layout: jobs | slot_off | rel_off | lens | prefix_off | prefix | preamble | results | digests | frame_len | frame_off | queue
  uint64_t mo = 0;
  auto place = [&](uint64_t bytes) { uint64_t o = mo; mo = align_up(mo + bytes, 256); return o; };
  const uint64_t o_jobs = place(sizeof(EncJob) * nb), o_slot = place(8ull * (nb + 1)), o_rel = place(8ull * (nb + 1)), o_preoff = place(8ull * (nb + 1)),
                 o_len = place(4ull * nb), o_poff = place(4ull * (nb + 1)), o_prefix = place(prefix.size()),
                 o_pre = place(preamble.size()), o_res = place(sizeof(BlockResult) * nb), o_dig = place(20ull * nb),
                 o_flen = place(8ull * nb), o_foff = place(8ull * (nb + 1)), o_queue = place(256);
  reserve_io(d.meta, mo, d.arena);
  uint8_t* meta = d.meta.as<uint8_t>();
  const uint8_t* d_in;
  if (T.d_in_ext) d_in = T.d_in_ext + in_base;
  else { reserve_io(d.in, std::max<uint64_t>(in_total, 16), d.arena); d_in = d.in.as<uint8_t>(); }
  uint8_t* d_work = nullptr;  // pre-processed copy when the transform must not touch the caller's data
  if (do_e8 && T.d_in_ext) { reserve_io(d.work, std::max<uint64_t>(in_total, 16), d.arena); d_work = d.work.as<uint8_t>(); }
  uint8_t* d_pre = nullptr;   // transformed streams (LZ77 / BWT output)
  if (lz_level) { reserve_io(d.pre, std::max<uint64_t>(pre_total, 16), d.arena); d_pre = d.pre.as<uint8_t>(); }
  reserve_io(d.slots, std::max<uint64_t>(slots_total, 16), d.arena);
  uint8_t* d_out = T.d_out_ext;
  if (!d_out) { reserve_io(d.out, std::max<uint64_t>(slots_total, 16), d.arena); d_out = d.out.as<uint8_t>(); }
  const uint64_t d_out_cap = T.d_out_ext ? T.d_out_cap : d.out.cap;

  // ---- launch geometry: arenas take what is left ----
  Launch L;
  if (M.hdr.n) {
    const uint64_t fr = free_device_memory() + d.arena.cap;
    const uint64_t reserve = 512ull << 20;
    // time-skewed encoder: every lane model whose coder delay fits (zpq_pipe.cuh); ZPQ_PIPE=0 keeps the
    // bit-by-bit lane encoder (A/B measurements); blocks of 2^28 bytes and more overflow its bit counter
    // ZPQ_DUO=0 keeps the single-warp encoders (A/B measurements)
    const char* e = getenv("ZPQ_PIPE");
    const char* e2 = getenv("ZPQ_DUO");
    const bool fits = max_block + max_block / 16 + preamble.size() + 64 < (1ull << 28);
    const bool want_skew = !(e && *e == '0') && fits;
    const bool want_duo = !(e2 && *e2 == '0') && fits;
    plan_launch(d, M.hdr, false, nb, fr > reserve ? fr - reserve : 0, ctx->max_resident, L, want_skew, want_duo, false,
                max_block + max_block / 16 + preamble.size() + 64);
    d.arena.reserve((uint64_t)L.resident * L.plan->arena_bytes);
  } else {
    plan_launch(d, M.hdr, false, nb, 1ull << 30, ctx->max_resident, L);
    d.arena.reserve(std::max<uint64_t>((uint64_t)L.resident * L.plan->arena_bytes, 4096));
  }
  // The state arenas are idle until the coding kernel starts, so the pre-processing scratch
  // (suffix-array workspace, SA / ISA, LZ77 hash tables) lives in the same memory.
  const uint64_t ht_entries = (lz_level == 1 || lz_level == 2) && !use_sa ? (1ull << M.args[5]) : 0;
  auto scratch_for = [&](uint64_t bytes, uint64_t blocks) -> uint64_t {
    uint64_t need = 4096;
    if (use_sa) need += sa_workspace_bytes(bytes) + 8 * bytes + 1024;      // workspace + SA + ISA
    need += ht_entries * 4 * blocks;
    return need;
  };
  if (lz_level) {
    const uint64_t want = scratch_for(in_total, nb);
    if (d.arena.cap < want) {
      const uint64_t fr = free_device_memory() + d.arena.cap;
      const uint64_t reserve = 512ull << 20;
      const uint64_t can = fr > reserve ? fr - reserve : 0;
      if (std::min(want, can) > d.arena.cap) d.arena.reserve(std::min(want, can));
    }
  }
  d.plan.reserve(sizeof(Plan));
  CU(cudaMemcpyAsync(d.plan.p, L.plan.get(), sizeof(Plan) - sizeof(L.plan->hcomp) + L.plan->hcomp_len + 8,
                     cudaMemcpyHostToDevice, s));

  // ---- uploads ----
  d.t_h2d.start(s);
  auto up = [&](uint64_t o, const void* src, uint64_t bytes) {
    if (bytes) CU(cudaMemcpyAsync(meta + o, src, bytes, cudaMemcpyHostToDevice, s));
  };
  up(o_jobs, jobs.data(), sizeof(EncJob) * nb);
  up(o_slot, slot_off.data(), 8ull * (nb + 1));
  up(o_rel, rel_off.data(), 8ull * (nb + 1));
  up(o_preoff, pre_off.data(), 8ull * (nb + 1));
  up(o_len, lens.data(), 4ull * nb);
  up(o_poff, prefix_off.data(), 4ull * (nb + 1));
  up(o_prefix, prefix.data(), prefix.size());
  up(o_pre, preamble.data(), preamble.size());
  CU(cudaMemsetAsync(meta + o_queue, 0, 256, s));
  if (!T.d_in_ext && in_total) {
    CU(cudaMemcpyAsync(d.in.p, T.h_in + in_base, in_total, cudaMemcpyHostToDevice, s));
    d.stats.h2d_bytes = in_total;
  }
  d.t_h2d.stop(s);

  // ---- kernels ----
  d.t_kern.start(s);
  uint32_t launches = 0;
  if (T.dosha1) {
    CU(launch_sha1(d_in, (const uint64_t*)(meta + o_rel), (const uint32_t*)(meta + o_len), nb, meta + o_dig, s));
    ++launches;
  }
  const uint8_t* d_coded_in = d_in;
  if (do_e8) {  // E8E9 after the checksum, LibZPAQ.cs:307-310 / LZBuffer.cs:198
    uint8_t* tgt = d_work ? d_work : const_cast<uint8_t*>(d_in);
    if (d_work) CU(cudaMemcpyAsync(d_work, d_in, in_total, cudaMemcpyDeviceToDevice, s));
    CU(launch_e8e9(tgt, (const uint64_t*)(meta + o_rel), (const uint32_t*)(meta + o_len), nb, s));
    d_coded_in = tgt;
    ++launches;
  }
  if (lz_level) {
    // chunks of consecutive blocks whose scratch fits in the arena memory
    const uint8_t* src = d_coded_in;
    uint32_t b0 = 0;
    while (b0 < nb) {
      uint32_t b1 = b0;
      uint64_t bytes = 0;
      while (b1 < nb) {
        const uint64_t nbytes = bytes + (off[b1 + 1] - off[b1]);
        if (b1 > b0 && (scratch_for(nbytes, b1 + 1 - b0) > d.arena.cap || nbytes >= (1ull << 32) - 4096)) break;
        bytes = nbytes; ++b1;
      }
      if (scratch_for(bytes, b1 - b0) > d.arena.cap) throw Failure(ZPQ_E_NOMEM, "pre-processing scratch does not fit in device memory");
      uint8_t* scratch = d.arena.as<uint8_t>();
      uint64_t so = 0;
      auto stake = [&](uint64_t n) { uint8_t* q = scratch + so; so = align_up(so + n, 256); return q; };
      uint32_t* sa = nullptr; uint32_t* isa = nullptr;
      const uint8_t* chunk_in = src + rel_off[b0];
      const uint64_t* chunk_off = (const uint64_t*)(meta + o_rel) + b0;
      uint64_t chunk_max = 0;
      for (uint32_t b = b0; b < b1; ++b) chunk_max = std::max<uint64_t>(chunk_max, off[b + 1] - off[b]);
      if (use_sa) {
        sa = (uint32_t*)stake(4 * bytes);
        isa = lz_level == 3 ? nullptr : (uint32_t*)stake(4 * bytes);
        const size_t wsb = sa_workspace_bytes(bytes);
        void* ws = stake(wsb);
        int rounds = 0;
        CU(build_suffix_arrays(chunk_in, chunk_off, b1 - b0, bytes, chunk_max, sa, isa, ws, wsb, s, &rounds));
        launches += 3 + 5 * rounds;
      }
      if (lz_level == 3) {
        CU(launch_bwt_emit(chunk_in, chunk_off, sa, (const uint64_t*)(meta + o_preoff) + b0, d_pre, (EncJob*)(meta + o_jobs) + b0,
                           b1 - b0, chunk_max, s));
      } else {
        LzParams Z{};
        Z.in = chunk_in; Z.off = chunk_off; Z.out = d_pre; Z.out_off = (const uint64_t*)(meta + o_preoff) + b0;
        Z.jobs = (EncJob*)(meta + o_jobs) + b0;
        Z.ht = ht_entries ? (uint32_t*)stake(ht_entries * 4 * (b1 - b0)) : nullptr;
        Z.sa = sa; Z.isa = isa; Z.nb = b1 - b0; Z.htsize = (uint32_t)ht_entries;
        Z.level = lz_level; Z.use_sa = use_sa ? 1 : 0;
        Z.checkbits = use_sa ? 17 + M.args[0] : 12 - M.args[0];
        if (Z.checkbits < 0 || Z.checkbits > 31) throw Failure(ZPQ_E_UNSUPPORTED, "LZ77 check bits out of range");
        Z.minMatch = M.args[2]; Z.minMatch2 = M.args[3];
        Z.maxMatch = (1u << 14) * 3; Z.maxLiteral = (1u << 14) / 4;
        Z.lookahead = M.args[6];
        Z.bucket = (1u << M.args[4]) - 1;
        Z.shift1 = Z.minMatch > 0 ? (M.args[5] - 1) / Z.minMatch + 1 : 1;
        Z.shift2 = Z.minMatch2 > 0 ? (M.args[5] - 1) / Z.minMatch2 + 1 : 0;
        Z.minMatchBoth = std::max(Z.minMatch, Z.minMatch2 + Z.lookahead) + 4;
        Z.rb = M.args[0] > 4 ? M.args[0] - 4 : 0;
        CU(launch_lz77(Z, s));
      }
      ++launches;
      b0 = b1;
    }
    d_coded_in = d_pre;
  }
  CodecParams P{};
  P.plan = d.plan.as<Plan>();
  P.tab = d.d_tab;
  P.arenas = d.arena.as<uint8_t>();
  P.arena_stride = L.plan->arena_bytes;
  P.in = d_coded_in;
  P.preamble = meta + o_pre;
  P.out = d.slots.as<uint8_t>();
  P.ejobs = (const EncJob*)(meta + o_jobs);
  P.results = (BlockResult*)(meta + o_res);
  P.njobs = nb;
  P.resident = L.resident;
  P.queue = (uint32_t*)(meta + o_queue);
  P.wb = L.wb;
  P.sm = L.sm;
  d.t_codec.start(s);
  CU(launch_codec(L, P, false, s));
  d.t_codec.stop(s);
  ++launches;

  FinishParams F{};
  F.slots = d.slots.as<uint8_t>();
  F.slot_off = (const uint64_t*)(meta + o_slot);
  F.prefix = meta + o_prefix;
  F.prefix_off = (const uint32_t*)(meta + o_poff);
  F.results = (const BlockResult*)(meta + o_res);
  F.digests = T.dosha1 ? meta + o_dig : nullptr;
  F.frame_len = (uint64_t*)(meta + o_flen);
  F.nb = nb;
  CU(launch_finish(F, s));
  CU(launch_scan((const uint64_t*)(meta + o_flen), (uint64_t*)(meta + o_foff), nb, s));
  CU(launch_gather(d.slots.as<uint8_t>(), (const uint64_t*)(meta + o_slot), (const uint64_t*)(meta + o_flen), d_out,
                   (const uint64_t*)(meta + o_foff), d_out_cap, nb, max_frame, s));
  launches += 3;
  d.t_kern.stop(s);

  // ---- results ----
  std::vector<BlockResult> res(nb);
  T.frame_off.assign(nb + 1, 0);
  d.t_d2h.start(s);
  CU(cudaMemcpyAsync(res.data(), meta + o_res, sizeof(BlockResult) * nb, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(T.frame_off.data(), meta + o_foff, 8ull * (nb + 1), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (uint32_t i = 0; i < nb; ++i) {
    if (res[i].status == ZPQ_BLOCK_OVERFLOW) throw Failure(ZPQ_E_OUTPUT, "coded block " + std::to_string(T.first + i) + " outgrew its slot");
    if (res[i].status != ZPQ_BLOCK_OK) throw Failure(ZPQ_E_CONFIG, "ZPAQL execution error while coding block " + std::to_string(T.first + i));
  }
  const uint64_t total = T.frame_off[nb];
  if (total > d_out_cap) throw Failure(ZPQ_E_OUTPUT, "output buffer too small");
  if (h_out) {
    if (total > h_out_cap) throw Failure(ZPQ_E_OUTPUT, "output buffer too small");
    CU(cudaMemcpyAsync(h_out, d_out, total, cudaMemcpyDeviceToHost, s));
    d.stats.d2h_bytes = total;
  }
  d.t_d2h.stop(s);
  d.t_all.stop(s);
  CU(cudaStreamSynchronize(s));
  d.stats.h2d_ms = d.t_h2d.ms(); d.stats.kernel_ms = d.t_kern.ms(); d.stats.d2h_ms = d.t_d2h.ms();
  d.stats.total_ms = d.t_all.ms(); d.stats.codec_kernel_ms = d.t_codec.ms();
  d.stats.launches = launches; d.stats.resident_blocks = L.resident; d.stats.state_bytes_per_block = L.plan->arena_bytes;
  snprintf(d.stats.kernel, sizeof d.stats.kernel, "%s", L.kernel.c_str());
  return total;
}

// Split [0, nb) among the context's devices by input bytes, run them concurrently, and lay the
// results out in block order.
void compress_model(zpq_ctx* ctx, const Model& M, const uint8_t* in, const uint64_t* in_off, uint32_t first, uint32_t nb,
                    const std::vector<std::string>& filenames, const std::vector<std::string>& comments, bool dosha1,
                    bool with_tag, uint8_t* out, uint64_t out_cap, uint64_t out_base, uint64_t* out_off) {
  const size_t nd = std::min<size_t>(ctx->devs.size(), std::max<uint32_t>(nb, 1));
  std::vector<uint32_t> cut(nd + 1, first);
  {
    const uint64_t total = in_off[first + nb] - in_off[first];
    uint32_t b = first;
    for (size_t k = 1; k < nd; ++k) {
      const uint64_t target = in_off[first] + total * k / nd;
      while (b < first + nb && in_off[b] < target) ++b;
      cut[k] = b;
    }
    cut[nd] = first + nb;
  }
  if (nd == 1) {
    CompressTask T;
    T.model = &M; T.h_in = in; T.in_off = in_off; T.first = first; T.count = nb;
    T.filenames = filenames; T.comments = comments; T.dosha1 = dosha1; T.with_tag = with_tag;
    if (out_base > out_cap) throw Failure(ZPQ_E_OUTPUT, "output buffer too small");
    compress_on_device(ctx, ctx->devs[0], T, out + out_base, out_cap - out_base);
    for (uint32_t i = 0; i <= nb; ++i) out_off[first + i] = out_base + T.frame_off[i];
    return;
  }
  // several devices: each compresses its range into its own device buffer and copies it to its final place as soon as
  // the devices in front of it have reported their sizes (ordered reassembly through asynchronous copies: a device's
  // D2H overlaps the kernels of the devices still running)
  std::vector<CompressTask> tasks(nd);
  std::vector<std::string> errs(nd);
  std::vector<int> codes(nd, 0);
  std::vector<std::thread> th;
  std::mutex mu;
  std::condition_variable cv;
  std::vector<int> done(nd, 0);
  std::vector<uint64_t> totals(nd, 0);
  for (size_t k = 0; k < nd; ++k) {
    CompressTask& T = tasks[k];
    T.model = &M; T.h_in = in; T.in_off = in_off; T.first = cut[k]; T.count = cut[k + 1] - cut[k];
    T.dosha1 = dosha1; T.with_tag = with_tag;
    for (uint32_t i = cut[k]; i < cut[k + 1]; ++i) {
      T.filenames.push_back(filenames.size() > i - first ? filenames[i - first] : std::string());
      T.comments.push_back(comments.size() > i - first ? comments[i - first] : std::string());
    }
    th.emplace_back([&, k]() {
      try {
        if (tasks[k].count) compress_on_device(ctx, ctx->devs[k], tasks[k], nullptr, 0);
        else tasks[k].frame_off.assign(1, 0);
        totals[k] = tasks[k].frame_off[tasks[k].count];
      } catch (const Failure& f) { codes[k] = f.code; errs[k] = f.what(); }
      catch (const std::exception& e) { codes[k] = ZPQ_E_CUDA; errs[k] = e.what(); }
      uint64_t base = out_base;
      {
        std::unique_lock<std::mutex> lk(mu);
        done[k] = 1;
        cv.notify_all();
        cv.wait(lk, [&]() { for (size_t j = 0; j < k; ++j) if (!done[j]) return false; return true; });
        for (size_t j = 0; j < k; ++j) base += totals[j];
      }
      if (codes[k]) return;
      const CompressTask& T = tasks[k];
      for (uint32_t i = 0; i <= T.count; ++i) out_off[T.first + i] = base + T.frame_off[i];
      if (base + totals[k] > out_cap) { codes[k] = ZPQ_E_OUTPUT; errs[k] = "output buffer too small"; return; }
      Device& d = ctx->devs[k];
      if (cudaSetDevice(d.id) != cudaSuccess || (totals[k] && cudaMemcpyAsync(out + base, d.out.p, totals[k], cudaMemcpyDeviceToHost, d.stream) != cudaSuccess) ||
          cudaStreamSynchronize(d.stream) != cudaSuccess) { codes[k] = ZPQ_E_CUDA; errs[k] = "copy of the archive to the host failed"; }
      d.stats.d2h_bytes = totals[k];
    });
  }
  for (auto& t : th) t.join();
  for (size_t k = 0; k < nd; ++k) if (codes[k]) throw Failure(codes[k], errs[k]);
}

// The data analysis of method levels 5..9 (LibZPAQ.cs:242-258) for every block of a batch, on device 0: byte-gap histograms,
// kGapBins ints per block.  The blocks go up in pieces of about 1 GB; the models are then derived on the host from 16 KB per block.
void device_gap_histograms(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, std::vector<int>& gaps) {
  Device& d = ctx->devs[0];
  CU(cudaSetDevice(d.id));
  cudaStream_t s = d.stream;
  gaps.assign((size_t)nb * kGapBins, 0);
  uint32_t b0 = 0;
  while (b0 < nb) {
    uint32_t b1 = b0 + 1;
    while (b1 < nb && in_off[b1 + 1] - in_off[b0] <= (1ull << 30)) ++b1;
    const uint32_t cnt = b1 - b0;
    const uint64_t bytes = in_off[b1] - in_off[b0];
    uint64_t max_len = 0;
    for (uint32_t b = b0; b < b1; ++b) max_len = std::max(max_len, in_off[b + 1] - in_off[b]);
    reserve_io(d.in, bytes + 64, d.arena);
    uint64_t mo = 0;
    auto place = [&](uint64_t n) { uint64_t o = mo; mo = align_up(mo + n, 256); return o; };
    const uint64_t o_off = place(8ull * (cnt + 1)), o_gap = place(4ull * cnt * kGapBins);
    d.meta.reserve(mo);
    uint8_t* meta = d.meta.as<uint8_t>();
    if (bytes) CU(cudaMemcpyAsync(d.in.p, in + in_off[b0], bytes, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(meta + o_off, in_off + b0, 8ull * (cnt + 1), cudaMemcpyHostToDevice, s));
    CU(launch_gap_hist(d.in.as<uint8_t>(), (const uint64_t*)(meta + o_off), cnt, max_len, (int*)(meta + o_gap), s));
    CU(cudaMemcpyAsync(gaps.data() + (size_t)b0 * kGapBins, meta + o_gap, 4ull * cnt * kGapBins, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    b0 = b1;
  }
}


void model_from_header_bytes(const uint8_t* hdr, uint64_t hdr_len, const uint8_t* pcomp, uint64_t pcomp_len, const int* args9,
                             Model& M) {
  if (!hdr || hdr_len < 8) throw Failure(ZPQ_E_ARG, "missing block header");
  size_t used = parse_header(hdr, hdr_len, M.hdr);
  if (used != hdr_len) throw Failure(ZPQ_E_ARG, "block header length mismatch");
  M.pcomp.assign(pcomp, pcomp + (pcomp ? pcomp_len : 0));
  if (M.pcomp.size() > 65535) throw Failure(ZPQ_E_ARG, "PCOMP program too long");
  for (int i = 0; i < 9; ++i) M.args[i] = args9 ? args9[i] : 0;
}

// ------------------------------------------------------------------------------------------
// Decompression
// ------------------------------------------------------------------------------------------
struct DecBlock {
  BlockRef ref;
  uint64_t start;      // absolute offset of the block in `in`
  uint64_t cap;        // output slot capacity
  bool hinted;
};

// ZPQ_FDEC=0 keeps the lane-resident decoders with the post-processor inside (A/B measurements)
bool want_fast_decode() { const char* e = getenv("ZPQ_FDEC"); return !(e && *e == '0'); }
// ZPQ_NATIVE_POST=0 sends every block through the PCOMP interpreter pass (test hook: both must restore the same bytes)
bool want_native_post() { const char* e = getenv("ZPQ_NATIVE_POST"); return !(e && *e == '0'); }

// Blocks [b0, b1) on one device: H2D of their archive bytes, decode (+ post-processing pass), SHA-1, ordered
// compaction into d.out.  Fills lens / bstat / sha for these blocks; the caller copies d.out to the host.
struct DecodeRange {
  uint32_t b0 = 0, b1 = 0;
  uint64_t total = 0;          // restored bytes of the range, gathered in d.out
  std::string first_err;
  bool any_corrupt = false;
};

void decompress_range(zpq_ctx* ctx, Device& d, std::vector<DecBlock>& blocks, DecodeRange& R, const uint8_t* in, const uint64_t* in_off,
                      std::vector<uint64_t>& lens, std::vector<uint8_t>& bstat, std::vector<uint8_t>& sha) {
  CU(cudaSetDevice(d.id));
  cudaStream_t s = d.stream;
  d.stats = zpq_stats{};
  d.t_all.start(s);
  const uint32_t b0 = R.b0, b1 = R.b1, nbr = b1 - b0;
  const uint64_t in_base = in_off[b0], in_total = in_off[b1] - in_off[b0];
  reserve_io(d.in, in_total + 64, d.arena);
  d.t_h2d.start(s);
  if (in_total) CU(cudaMemcpyAsync(d.in.p, in + in_base, in_total, cudaMemcpyHostToDevice, s));
  d.stats.h2d_bytes = in_total;
  d.t_h2d.stop(s);

  std::vector<BlockResult> res(nbr);
  std::vector<uint32_t> pending;
  for (uint32_t i = b0; i < b1; ++i) if (bstat[i] == ZPQ_BLOCK_OK) pending.push_back(i);
  std::vector<uint64_t> slot_off(nbr + 1, 0);
  std::vector<std::vector<uint64_t>> seg_out(nbr);      // restored bytes of a block at the end of each of its segments
  std::atomic<uint32_t> launches{0};
  double codec_ms = 0, post_ms = 0;
  uint32_t post_native = 0, post_interp = 0, post_compiled = 0;
  d.t_kern.start(s);
  auto fail_block = [&](uint32_t i, uint8_t st, const std::string& why) {
    bstat[i] = st; R.any_corrupt = true;
    if (R.first_err.empty()) R.first_err = "block " + std::to_string(i) + ": " + why;
  };
  // Slots of finished blocks stay where they are; a block that outgrew its slot gets a larger one behind them and is
  // decoded again (the size in a segment comment is only a first guess: the reference ignores comments, LibZPAQ.cs:65-79).
  uint64_t slots_total = 0;
  for (int attempt = 0; attempt < 8 && !pending.empty(); ++attempt) {
    uint64_t need = slots_total;
    for (uint32_t i : pending) { slot_off[i - b0] = need; need = align_up(need + blocks[i].cap, 16); }
    if (need > d.slots.cap) {
      // grow, keeping what finished blocks already hold
      DevBuf bigger;
      const uint64_t fr = free_device_memory();
      if (need > fr + d.arena.cap) {
        for (uint32_t i : pending) fail_block(i, ZPQ_BLOCK_OVERFLOW, "restored data does not fit in device memory");
        pending.clear();
        break;
      }
      try { bigger.reserve(need); }
      catch (const Failure&) { cudaGetLastError(); d.arena.release(); bigger.reserve(need); }
      if (slots_total) CU(cudaMemcpyAsync(bigger.p, d.slots.p, slots_total, cudaMemcpyDeviceToDevice, s));
      CU(cudaStreamSynchronize(s));
      d.slots.release();
      d.slots = bigger; bigger.p = nullptr; bigger.cap = 0;
    }
    slots_total = need;
    // group by header bytes
    std::map<Bytes, std::vector<uint32_t>> groups;
    for (uint32_t i : pending) groups[blocks[i].ref.hdr.wire].push_back(i);
    std::mutex alloc_mu, res_mu;
    auto run_group = [&](const std::vector<uint32_t>& ids, GroupBufs G, bool may_defer, GroupBarrier* bar) {
      const Header& hdr = blocks[ids[0]].ref.hdr;
      bool arrived = false;
      try {
        std::vector<DecJob> jobs(ids.size());
        std::vector<PostJob> pjobs(ids.size());
        std::vector<DecSeg> segs;
        // every decoder leaves the raw model stream -- PCOMP preamble (<= 64 KB + 3) + transformed data (LZ77 output may
        // exceed the data by 1/16) -- in G.work; the post-processing pass turns it into the restored bytes in the slots
        uint64_t raw_total = 0, max_raw = 0;
        for (size_t k = 0; k < ids.size(); ++k) {
          const DecBlock& b = blocks[ids[k]];
          jobs[k].seg_first = (uint32_t)segs.size();
          jobs[k].seg_count = (uint32_t)b.ref.segs.size();
          pjobs[k].out_off = slot_off[ids[k] - b0];
          pjobs[k].out_cap = b.cap;
          jobs[k].out_off = raw_total; jobs[k].out_cap = b.cap + b.cap / 8 + 70000;
          max_raw = std::max(max_raw, jobs[k].out_cap);
          raw_total = align_up(raw_total + jobs[k].out_cap, 16);
          for (const SegmentRef& sg : b.ref.segs) segs.push_back(DecSeg{b.start - in_base + sg.data_off, sg.data_len});
        }
        std::unique_lock<std::mutex> alloc_lk(alloc_mu);    // groups size and take their memory one after the other, then run side by side
        reserve_io(G.work, std::max<uint64_t>(raw_total, 16) + 64, G.arena);       // before the arenas are sized
        std::vector<PostCandidate> cands;
        post_candidates(hdr.ph, hdr.pm, cands);
        std::vector<PostCand> dcands(cands.size());
        Bytes cand_bytes;
        bool has_bwt = false;
        for (size_t k = 0; k < cands.size(); ++k) {
          dcands[k] = PostCand{cands[k].kind, cands[k].e8, cands[k].param, (uint32_t)cand_bytes.size(), (uint32_t)cands[k].prog.size(), cands[k].wild};
          cand_bytes.insert(cand_bytes.end(), cands[k].prog.begin(), cands[k].prog.end());
          has_bwt = has_bwt || cands[k].kind == PK_BWT;
        }
        Launch L;
        const uint64_t fr = free_device_memory() + G.arena.cap;
        const uint64_t reserve = 512ull << 20;
        plan_launch(d, hdr, true, ids.size(), fr > reserve ? fr - reserve : 0, ctx->max_resident, L, false, false, want_fast_decode(), max_raw);
        uint64_t mo = 0;
        auto place = [&](uint64_t bytes) { uint64_t o = mo; mo = align_up(mo + bytes, 256); return o; };
        const size_t nseg = std::max<size_t>(segs.size(), 1);
        const uint64_t o_jobs = place(sizeof(DecJob) * jobs.size()), o_segs = place(sizeof(DecSeg) * nseg), o_send = place(8ull * nseg),
                       o_pjobs = place(sizeof(PostJob) * jobs.size()), o_raw = place(sizeof(BlockResult) * jobs.size()),
                       o_res = place(sizeof(BlockResult) * jobs.size()), o_queue = place(512), o_kind = place(4ull * jobs.size()),
                       o_cand = place(sizeof(PostCand) * std::max<size_t>(dcands.size(), 1)), o_cbytes = place(cand_bytes.size() + 16),
                       o_sout = place(8ull * nseg);
        G.meta.reserve(mo);
        uint8_t* meta = G.meta.as<uint8_t>();
        G.arena.reserve((uint64_t)L.resident * L.plan->arena_bytes);
        G.plan.reserve(sizeof(Plan));
        alloc_lk.unlock();
        if (bar) { arrived = true; bar->arrive_and_wait(); }
        CU(cudaMemcpyAsync(G.plan.p, L.plan.get(), sizeof(Plan) - sizeof(L.plan->hcomp) + L.plan->hcomp_len + 8,
                           cudaMemcpyHostToDevice, G.stream));
        CU(cudaMemcpyAsync(meta + o_jobs, jobs.data(), sizeof(DecJob) * jobs.size(), cudaMemcpyHostToDevice, G.stream));
        CU(cudaMemcpyAsync(meta + o_pjobs, pjobs.data(), sizeof(PostJob) * jobs.size(), cudaMemcpyHostToDevice, G.stream));
        if (!segs.empty()) CU(cudaMemcpyAsync(meta + o_segs, segs.data(), sizeof(DecSeg) * segs.size(), cudaMemcpyHostToDevice, G.stream));
        if (!dcands.empty()) {
          CU(cudaMemcpyAsync(meta + o_cand, dcands.data(), sizeof(PostCand) * dcands.size(), cudaMemcpyHostToDevice, G.stream));
          CU(cudaMemcpyAsync(meta + o_cbytes, cand_bytes.data(), cand_bytes.size(), cudaMemcpyHostToDevice, G.stream));
        }
        CU(cudaMemsetAsync(meta + o_queue, 0, 512, G.stream));
        CU(cudaMemsetAsync(meta + o_sout, 0, 8ull * nseg, G.stream));
        CodecParams P{};
        P.plan = G.plan.as<Plan>(); P.tab = d.d_tab;
        P.arenas = G.arena.as<uint8_t>(); P.arena_stride = L.plan->arena_bytes;
        P.in = d.in.as<uint8_t>(); P.out = G.work.as<uint8_t>();
        P.djobs = (const DecJob*)(meta + o_jobs); P.segs = (const DecSeg*)(meta + o_segs);
        P.seg_end = (uint64_t*)(meta + o_send);
        P.results = (BlockResult*)(meta + o_raw);
        P.njobs = (uint32_t)jobs.size(); P.resident = L.resident; P.queue = (uint32_t*)(meta + o_queue); P.sm = L.sm;
        G.t_codec.start(s);
        CU(launch_codec(L, P, true, G.stream));
        G.t_codec.stop(s);
        ++launches;
        {
          PostParams Q{};
          Q.plan = G.plan.as<Plan>(); Q.arenas = G.arena.as<uint8_t>(); Q.arena_stride = L.plan->arena_bytes;
          Q.raw = G.work.as<uint8_t>(); Q.djobs = P.djobs; Q.seg_end = P.seg_end; Q.raw_results = (const BlockResult*)(meta + o_raw);
          Q.out = d.slots.as<uint8_t>(); Q.pjobs = (const PostJob*)(meta + o_pjobs); Q.results = (BlockResult*)(meta + o_res);
          Q.njobs = P.njobs; Q.resident = L.resident; Q.queue = (uint32_t*)(meta + o_queue + 256); Q.queue2 = (uint32_t*)(meta + o_queue + 128);
          Q.jobkind = (uint32_t*)(meta + o_kind); Q.seg_out_end = (uint64_t*)(meta + o_sout);
          Q.cand_bytes = meta + o_cbytes; Q.cands = (const PostCand*)(meta + o_cand); Q.ncand = (uint32_t)dcands.size();
          Q.has_bwt = has_bwt ? 1u : 0u; Q.max_raw = max_raw;
          G.t_post.start(s);
          if (want_native_post()) { CU(launch_post_native(Q, G.stream)); launches += 4; }
          else CU(cudaMemsetAsync(meta + o_kind, 0, 4ull * jobs.size(), G.stream));
          // Blocks left over (foreign programs; streams a native kernel handed back): their stored program is translated to
          // C and compiled with NVRTC for sm_100a -- one kernel per distinct program, at most four per batch -- and whatever
          // that does not take is interpreted.
          {
            std::vector<uint32_t> kd(jobs.size());
            std::vector<BlockResult> rr(jobs.size());
            std::vector<Bytes> tried;
            for (int round = 0; round < 4; ++round) {
              CU(cudaMemcpyAsync(kd.data(), meta + o_kind, 4ull * jobs.size(), cudaMemcpyDeviceToHost, G.stream));
              if (round == 0) CU(cudaMemcpyAsync(rr.data(), meta + o_raw, sizeof(BlockResult) * jobs.size(), cudaMemcpyDeviceToHost, G.stream));
              CU(cudaStreamSynchronize(G.stream));
              Bytes prog;
              for (size_t k = 0; k < jobs.size() && prog.empty(); ++k) {
                if ((kd[k] & 15u) != PK_GENERIC || rr[k].status != ZPQ_BLOCK_OK || rr[k].out_len < 4) continue;   // (damaged blocks: the interpreter pass reports them)
                uint8_t h3[3] = {0, 0, 0};
                CU(cudaMemcpy(h3, G.work.as<uint8_t>() + jobs[k].out_off, 3, cudaMemcpyDeviceToHost));
                const uint32_t psize = h3[1] + 256u * h3[2];
                if (h3[0] != 1 || psize < 1 || 3ull + psize > rr[k].out_len || psize > 8192) continue;              // (huge programs are not worth a compile)
                Bytes pg(psize);
                CU(cudaMemcpy(pg.data(), G.work.as<uint8_t>() + jobs[k].out_off + 3, psize, cudaMemcpyDeviceToHost));
                if (std::find(tried.begin(), tried.end(), pg) == tried.end()) prog.swap(pg);
              }
              if (prog.empty()) break;
              tried.push_back(prog);
              std::string why;
              const void* kern = find_post_kernel(prog, hdr.ph, hdr.pm, &why);
              if (!kern) continue;
              const uint64_t o_prog = 0;
              DevBuf pbuf;                                     // program bytes + job counter; lives until the sync below
              pbuf.reserve(align_up(prog.size(), 256) + 256);
              CU(cudaMemcpyAsync(pbuf.as<uint8_t>() + o_prog, prog.data(), prog.size(), cudaMemcpyHostToDevice, G.stream));
              CU(cudaMemsetAsync(pbuf.as<uint8_t>() + align_up(prog.size(), 256), 0, 256, G.stream));
              const uint8_t* d_prog = pbuf.as<uint8_t>();
              uint32_t plen = (uint32_t)prog.size();
              uint32_t* d_cnt = (uint32_t*)(pbuf.as<uint8_t>() + align_up(prog.size(), 256));
              void* args[] = {&Q, &d_prog, &plen, &d_cnt};
              const uint32_t warps = std::min<uint32_t>(Q.resident, Q.njobs);
              CU(cudaLaunchKernel(kern, dim3((warps + 3) / 4), dim3(128), args, 0, G.stream));
              ++launches;
              CU(cudaStreamSynchronize(G.stream));
              pbuf.release();
            }
          }
          CU(launch_post(Q, G.stream));
          G.t_post.stop(s);
          ++launches;
        }
        std::vector<BlockResult> r(jobs.size());
        std::vector<uint32_t> kinds(jobs.size());
        std::vector<uint64_t> sout(nseg, 0);
        CU(cudaMemcpyAsync(sout.data(), meta + o_sout, 8ull * nseg, cudaMemcpyDeviceToHost, G.stream));
        CU(cudaMemcpyAsync(r.data(), meta + o_res, sizeof(BlockResult) * jobs.size(), cudaMemcpyDeviceToHost, G.stream));
        CU(cudaMemcpyAsync(kinds.data(), meta + o_kind, 4ull * jobs.size(), cudaMemcpyDeviceToHost, G.stream));
        CU(cudaStreamSynchronize(G.stream));
        std::lock_guard<std::mutex> res_lk(res_mu);
        for (uint32_t kd : kinds) { if ((kd & 15u) == PK_GENERIC) ++post_interp; else if ((kd & 15u) == PK_COMPILED) ++post_compiled; else ++post_native; }
        codec_ms += G.t_codec.ms();
        post_ms += G.t_post.ms();
        d.stats.resident_blocks = L.resident; d.stats.state_bytes_per_block = L.plan->arena_bytes;
        snprintf(d.stats.kernel, sizeof d.stats.kernel, "%s", L.kernel.c_str());
        for (size_t k = 0; k < ids.size(); ++k) {
          res[ids[k] - b0] = r[k];
          seg_out[ids[k] - b0].assign(sout.begin() + jobs[k].seg_first, sout.begin() + jobs[k].seg_first + jobs[k].seg_count);
        }
      } catch (const Failure& f) {
        if (bar && !arrived) { arrived = true; bar->arrive(); }
        // a header this build cannot run (or that does not fit) takes its own blocks down, not the batch
        if (f.code == ZPQ_E_CUDA) throw;
        if (f.code == ZPQ_E_NOMEM && may_defer) throw;          // no room beside the other groups: it runs alone afterwards
        cudaGetLastError();
        std::lock_guard<std::mutex> res_lk(res_mu);
        for (uint32_t i : ids) { res[i - b0].status = ZPQ_BLOCK_CORRUPT; res[i - b0].out_len = 0; fail_block(i, ZPQ_BLOCK_CORRUPT, f.what()); }
      } catch (...) {
        if (bar && !arrived) bar->arrive();
        throw;
      }
    };
    // Side by side only when the groups together leave SMs free: a batch with thousands of blocks fills every SM with the first
    // group's CTAs anyway, and the CTAs of the other groups queued between them only lengthen the tail (measured on the C5
    // archives: 1024 blocks of 1 MB 121 -> 176 MB/s, 256 blocks of 4 MB 33 -> 66 MB/s, but 4096 blocks of 256 kB 395 -> 280 MB/s).
    const bool side_by_side = groups.size() > 1 && pending.size() <= (size_t)d.sms * 8;
    if (!side_by_side) {
      for (auto& sc : d.pool) sc->release();                     // (a one-model batch may need all of HBM)
      for (auto& g : groups) run_group(g.second, GroupBufs{d.work, d.meta, d.plan, d.arena, s, d.t_codec, d.t_post}, false, nullptr);
    } else {
      // several models in the batch: one host thread and one stream per group (a group is a handful of latency-bound kernels;
      // run one after the other they would each wait for the longest chain of the one before)
      while (d.pool.size() + 1 < groups.size()) { d.pool.emplace_back(new Scratch); d.pool.back()->init(); }
      CU(cudaStreamSynchronize(s));
      if (free_device_memory() < (16ull << 30)) d.arena.release();   // an earlier one-model call left all of HBM there
      CU(cudaEventRecord(d.ev_ready, s));
      GroupBarrier bar;
      bar.need = groups.size();
      std::vector<std::thread> th;
      std::vector<std::string> terr(groups.size());
      std::vector<int> tcode(groups.size(), 0);
      size_t gi = 0;
      for (auto& g : groups) {
        const size_t k = gi++;
        th.emplace_back([&, k]() {
          bool entered = false;                                  // run_group always reaches the barrier once entered
          try {
            CU(cudaSetDevice(d.id));
            if (k == 0) { entered = true; run_group(g.second, GroupBufs{d.work, d.meta, d.plan, d.arena, s, d.t_codec, d.t_post}, true, &bar); }
            else {
              Scratch& sc = *d.pool[k - 1];
              CU(cudaStreamWaitEvent(sc.stream, d.ev_ready, 0));
              entered = true;
              run_group(g.second, GroupBufs{sc.work, sc.meta, sc.plan, sc.arena, sc.stream, sc.t_codec, sc.t_post}, true, &bar);
            }
          } catch (const Failure& f) { tcode[k] = f.code; terr[k] = f.what(); if (!entered) bar.arrive(); }
          catch (const std::exception& e) { tcode[k] = ZPQ_E_CUDA; terr[k] = e.what(); if (!entered) bar.arrive(); }
        });
      }
      for (auto& t : th) t.join();
      for (size_t k = 0; k < groups.size(); ++k) if (tcode[k] && tcode[k] != ZPQ_E_NOMEM) throw Failure(tcode[k], terr[k]);
      gi = 0;
      for (auto& g : groups) {                                   // groups that found no room beside the others: one at a time
        if (tcode[gi++] != ZPQ_E_NOMEM) continue;
        cudaGetLastError();
        for (auto& sc : d.pool) sc->release();
        run_group(g.second, GroupBufs{d.work, d.meta, d.plan, d.arena, s, d.t_codec, d.t_post}, false, nullptr);
      }
    }
    std::vector<uint32_t> again;
    for (uint32_t i : pending)
      if (bstat[i] == ZPQ_BLOCK_OK && res[i - b0].status == ZPQ_BLOCK_OVERFLOW) { blocks[i].cap = blocks[i].cap * 8 + (1 << 20); again.push_back(i); }
    pending.swap(again);
  }
  for (uint32_t i : pending) res[i - b0].status = ZPQ_BLOCK_OVERFLOW;
  // ---- SHA-1 of every SEGMENT's restored bytes, compared with the one stored behind the segment (Decompresser.readSegmentEnd,
  //      Decompresser.cs:163-194; LibZPAQ.decompress hashes per segment, LibZPAQ.cs:70-76) ----
  for (uint32_t i = b0; i < b1; ++i) {
    if (bstat[i] != ZPQ_BLOCK_OK) continue;
    bstat[i] = (uint8_t)res[i - b0].status;
    if (res[i - b0].status == ZPQ_BLOCK_OK) lens[i] = res[i - b0].out_len;
    else fail_block(i, (uint8_t)res[i - b0].status, "failed to decode (status " + std::to_string(res[i - b0].status) + ")");
  }
  {
    std::vector<uint64_t> h_soff;       // one range per segment that stores a checksum
    std::vector<uint32_t> h_slen, h_sblk, h_sseg;
    for (uint32_t i = 0; i < nbr; ++i) {
      if (bstat[b0 + i] != ZPQ_BLOCK_OK) continue;
      const auto& segs = blocks[b0 + i].ref.segs;
      const auto& ends = seg_out[i];
      uint64_t prev = 0;
      for (size_t k = 0; k < segs.size() && k < ends.size(); ++k) {
        const uint64_t end = std::min<uint64_t>(std::max(ends[k], prev), lens[b0 + i]);
        if (segs[k].has_sha1) { h_soff.push_back(slot_off[i] + prev); h_slen.push_back((uint32_t)(end - prev)); h_sblk.push_back(i); h_sseg.push_back((uint32_t)k); }
        prev = end;
      }
    }
    const uint32_t nsha = (uint32_t)h_soff.size();
    uint64_t mo = 0;
    auto place = [&](uint64_t bytes) { uint64_t o = mo; mo = align_up(mo + bytes, 256); return o; };
    const uint64_t o_slot = place(8ull * (nbr + 1)), o_len64 = place(8ull * nbr), o_foff = place(8ull * (nbr + 1)),
                   o_soff = place(8ull * std::max(nsha, 1u)), o_slen = place(4ull * std::max(nsha, 1u)), o_dig = place(20ull * std::max(nsha, 1u));
    d.meta.reserve(mo);
    uint8_t* meta = d.meta.as<uint8_t>();
    std::vector<uint64_t> len64(nbr);
    uint64_t max_len = 0, total = 0;
    for (uint32_t i = 0; i < nbr; ++i) { len64[i] = lens[b0 + i]; max_len = std::max(max_len, len64[i]); total += len64[i]; }
    reserve_io(d.slots, 16, d.arena);
    CU(cudaMemcpyAsync(meta + o_slot, slot_off.data(), 8ull * (nbr + 1), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(meta + o_len64, len64.data(), 8ull * nbr, cudaMemcpyHostToDevice, s));
    if (nsha) {
      CU(cudaMemcpyAsync(meta + o_soff, h_soff.data(), 8ull * nsha, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(meta + o_slen, h_slen.data(), 4ull * nsha, cudaMemcpyHostToDevice, s));
      CU(launch_sha1(d.slots.as<uint8_t>(), (const uint64_t*)(meta + o_soff), (const uint32_t*)(meta + o_slen), nsha, meta + o_dig, s));
    }
    CU(launch_scan((const uint64_t*)(meta + o_len64), (uint64_t*)(meta + o_foff), nbr, s));
    reserve_io(d.out, std::max<uint64_t>(total, 16), d.arena);
    CU(launch_gather(d.slots.as<uint8_t>(), (const uint64_t*)(meta + o_slot), (const uint64_t*)(meta + o_len64),
                     d.out.as<uint8_t>(), (const uint64_t*)(meta + o_foff), d.out.cap, nbr, max_len, s));
    launches += 3;
    d.t_kern.stop(s);
    std::vector<uint8_t> dig(20ull * std::max(nsha, 1u));
    if (nsha) CU(cudaMemcpyAsync(dig.data(), meta + o_dig, 20ull * nsha, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    // per block: 0 = no checksum stored, 1 = every stored checksum matched, 2 = at least one did not
    for (uint32_t i = 0; i < nbr; ++i) sha[b0 + i] = 0;
    for (uint32_t q = 0; q < nsha; ++q) {
      const uint32_t i = h_sblk[q];
      const bool same = memcmp(blocks[b0 + i].ref.segs[h_sseg[q]].sha1, &dig[20ull * q], 20) == 0;
      if (!same) sha[b0 + i] = 2;
      else if (sha[b0 + i] == 0) sha[b0 + i] = 1;
    }
    R.total = total;
  }
  d.stats.kernel_ms = d.t_kern.ms(); d.stats.h2d_ms = d.t_h2d.ms();
  d.stats.codec_kernel_ms = codec_ms; d.stats.post_kernel_ms = post_ms; d.stats.launches = launches;
  d.stats.post_native_blocks = post_native; d.stats.post_interpreted_blocks = post_interp; d.stats.post_compiled_blocks = post_compiled;
}

void decompress_all(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, uint8_t* out, uint64_t out_cap,
                    uint64_t* out_off, uint8_t* sha1_status, uint8_t* block_status) {
  // ---- parse framing on the host ----
  std::vector<DecBlock> blocks(nb);
  std::vector<uint8_t> bstat(nb, ZPQ_BLOCK_OK), sha(nb, 0);
  std::vector<uint64_t> lens(nb, 0);
  bool any_corrupt = false;
  std::string first_err;
  // (finding the end of a segment means looking at every coded byte, Decoder.cs:70-98: the blocks are parsed by all host cores)
  std::vector<std::string> perr(nb);
  auto parse_one = [&](uint32_t i) {
    DecBlock& b = blocks[i];
    b.start = in_off[i];
    try {
      parse_block(in + in_off[i], in_off[i + 1] - in_off[i], b.ref);
    } catch (const Failure& f) {
      bstat[i] = ZPQ_BLOCK_CORRUPT;
      perr[i] = "block " + std::to_string(i) + ": " + f.what();
      b.ref.segs.clear();
    }
    uint64_t cap = 0; b.hinted = true;
    for (const SegmentRef& sg : b.ref.segs) {
      // the decimal size a comment starts with is a hint only (the reference ignores comments on decode):
      // it is trusted as a first slot size while it is plausible for the coded bytes behind it
      const uint64_t guess = sg.data_len * 16 + (1 << 20);
      if (sg.size_hint >= 0 && (uint64_t)sg.size_hint <= std::max<uint64_t>(64ull << 20, sg.data_len * 4096)) cap += (uint64_t)sg.size_hint;
      else { b.hinted = false; cap += guess; }
    }
    b.cap = cap + 16;
  };
  {
    const uint32_t nt = (uint32_t)std::min<uint64_t>({(uint64_t)std::max(1u, std::thread::hardware_concurrency()), 32ull, (uint64_t)std::max<uint32_t>(nb, 1),
                                                      std::max<uint64_t>(1, (in_off[nb] - in_off[0]) >> 20)});
    if (nt <= 1) for (uint32_t i = 0; i < nb; ++i) parse_one(i);
    else {
      std::atomic<uint32_t> next{0};
      std::vector<std::thread> th;
      for (uint32_t t = 0; t < nt; ++t)
        th.emplace_back([&]() { for (;;) { const uint32_t i = next.fetch_add(1); if (i >= nb) break; parse_one(i); } });
      for (auto& t : th) t.join();
    }
    for (uint32_t i = 0; i < nb; ++i)
      if (!perr[i].empty()) { any_corrupt = true; if (first_err.empty()) first_err = perr[i]; }
  }
  // ---- partition over the devices by archive bytes, one host thread per device ----
  const size_t nd = std::min<size_t>(ctx->devs.size(), std::max<uint32_t>(nb, 1));
  std::vector<DecodeRange> ranges(nd);
  {
    const uint64_t total = in_off[nb] - in_off[0];
    uint32_t b = 0;
    for (size_t k = 0; k < nd; ++k) {
      ranges[k].b0 = b;
      if (k + 1 == nd) b = nb;
      else { const uint64_t target = in_off[0] + total * (k + 1) / nd; while (b < nb && in_off[b + 1] <= target) ++b; }
      ranges[k].b1 = b;
    }
  }
  std::vector<std::string> errs(nd);
  std::vector<int> codes(nd, 0);
  // device k copies its restored bytes out as soon as devices 0..k-1 have reported their totals (ordered reassembly
  // through asynchronous copies; no device waits for a slower one before starting its own kernels)
  std::mutex mu;
  std::condition_variable cv;
  std::vector<int> done(nd, 0);
  bool too_small = false;
  auto run = [&](size_t k) {
    DecodeRange& R = ranges[k];
    Device& d = ctx->devs[k];
    try {
      if (R.b1 > R.b0) decompress_range(ctx, d, blocks, R, in, in_off, lens, bstat, sha);
    } catch (const Failure& f) { codes[k] = f.code; errs[k] = f.what(); }
    catch (const std::exception& e) { codes[k] = ZPQ_E_CUDA; errs[k] = e.what(); }
    uint64_t base = 0;
    {
      std::unique_lock<std::mutex> lk(mu);
      done[k] = 1;
      cv.notify_all();
      cv.wait(lk, [&]() { for (size_t j = 0; j < k; ++j) if (!done[j]) return false; return true; });
      for (size_t j = 0; j < k; ++j) base += ranges[j].total;
    }
    if (codes[k] || R.b1 == R.b0) return;
    try {
      cudaStream_t s = d.stream;
      CU(cudaSetDevice(d.id));
      d.t_d2h.start(s);
      if (base + R.total > out_cap) { std::lock_guard<std::mutex> lk(mu); too_small = true; }
      else if (R.total) CU(cudaMemcpyAsync(out + base, d.out.p, R.total, cudaMemcpyDeviceToHost, s));
      d.stats.d2h_bytes = R.total;
      d.t_d2h.stop(s);
      d.t_all.stop(s);
      CU(cudaStreamSynchronize(s));
      d.stats.d2h_ms = d.t_d2h.ms(); d.stats.total_ms = d.t_all.ms();
    } catch (const Failure& f) { codes[k] = f.code; errs[k] = f.what(); }
  };
  if (nd == 1) run(0);
  else {
    std::vector<std::thread> th;
    for (size_t k = 0; k < nd; ++k) th.emplace_back(run, k);
    for (auto& t : th) t.join();
  }
  for (size_t k = 0; k < nd; ++k) if (codes[k]) throw Failure(codes[k], errs[k]);
  uint64_t acc = 0;
  for (uint32_t i = 0; i < nb; ++i) { out_off[i] = acc; acc += lens[i]; }
  out_off[nb] = acc;
  if (sha1_status) memcpy(sha1_status, sha.data(), nb);
  if (block_status) memcpy(block_status, bstat.data(), nb);
  if (too_small) throw Failure(ZPQ_E_OUTPUT, "output buffer too small");
  for (size_t k = 0; k < nd; ++k)
    if (ranges[k].any_corrupt) { any_corrupt = true; if (first_err.empty()) first_err = ranges[k].first_err; }
  if (any_corrupt) throw Failure(ZPQ_E_CORRUPT, first_err);
}

template <class F> int guarded(zpq_ctx* ctx, F&& f) {
  try { f(); return ZPQ_OK; }
  catch (const Failure& e) { if (ctx) ctx->err = e.what(); else { std::lock_guard<std::mutex> g(g_create_mutex); g_create_error = e.what(); } return e.code; }
  catch (const std::bad_alloc&) { if (ctx) ctx->err = "out of host memory"; return ZPQ_E_NOMEM; }
  catch (const std::exception& e) { if (ctx) ctx->err = e.what(); return ZPQ_E_CUDA; }
}

int64_t copy_out(const std::string& s, char* out, uint64_t cap) {
  if (out && cap) {
    const size_t k = std::min<size_t>(s.size(), cap - 1);
    memcpy(out, s.data(), k);
    out[k] = 0;
  }
  return (int64_t)s.size();
}

// ------------------------------------------------------------------------------------------
// Encryption (libzpaq AES_CTR): the key schedule is expanded on the host and wiped when the call returns.
// ------------------------------------------------------------------------------------------
constexpr uint64_t kAesChunk = 1ull << 30;   // device bytes per device for a host-buffer call

struct ScopedKey {
  AesKey k;
  ScopedKey(const uint8_t* key, int keylen) {
    if (!key || (keylen != 16 && keylen != 24 && keylen != 32)) throw Failure(ZPQ_E_ARG, "AES key length must be 16, 24 or 32 bytes");
    aes_expand_key(key, keylen, k);
  }
  ~ScopedKey() { secure_zero(&k, sizeof k); }
  std::string name() const { return "aes_ctr/" + std::to_string(32 * (k.rounds - 6)); }
};

void check_aes_range(const uint8_t* buf, uint64_t n, uint64_t offset) {
  if (!buf && n) throw Failure(ZPQ_E_ARG, "null buffer");
  if (n && offset > ~0ull - n) throw Failure(ZPQ_E_ARG, "offset + n overflows the 64-bit stream position");
}

// Bytes [0, n) of a host buffer, stream offset `offset`, through one device in chunks of kAesChunk: copy in, kernel, copy
// back.  A chunk lands at device address base + offset % 16, so its whole keystream blocks are 16-byte aligned.
void aes_ctr_host_range(Device& d, const ScopedKey& key, const uint8_t* iv8, uint8_t* buf, uint64_t n, uint64_t offset) {
  CU(cudaSetDevice(d.id));
  cudaStream_t s = d.stream;
  d.stats = zpq_stats{};
  snprintf(d.stats.kernel, sizeof d.stats.kernel, "%s", key.name().c_str());
  if (!n) return;
  const uint64_t chunk = std::min<uint64_t>(n, kAesChunk);
  reserve_io(d.in, chunk + 16, d.arena);
  d.t_all.start(s);
  for (uint64_t done = 0; done < n;) {
    const uint64_t len = std::min<uint64_t>(n - done, kAesChunk), off = offset + done;
    uint8_t* dev = d.in.as<uint8_t>() + off % 16;
    d.t_h2d.start(s);
    CU(cudaMemcpyAsync(dev, buf + done, len, cudaMemcpyHostToDevice, s));
    d.t_h2d.stop(s);
    d.t_kern.start(s);
    CU(launch_aes_ctr(key.k, iv8, dev, len, off, s));
    d.t_kern.stop(s);
    d.t_d2h.start(s);
    CU(cudaMemcpyAsync(buf + done, dev, len, cudaMemcpyDeviceToHost, s));
    d.t_d2h.stop(s);
    CU(cudaStreamSynchronize(s));
    d.stats.h2d_ms += d.t_h2d.ms(); d.stats.kernel_ms += d.t_kern.ms(); d.stats.d2h_ms += d.t_d2h.ms();
    d.stats.h2d_bytes += len; d.stats.d2h_bytes += len; d.stats.launches += 1;
    done += len;
  }
  d.t_all.stop(s);
  CU(cudaStreamSynchronize(s));
  d.stats.total_ms = d.t_all.ms();
}

// Split [0, n) into one contiguous byte range per device; every range carries its own stream offset, so the devices never
// exchange anything.
void aes_ctr_host(zpq_ctx* ctx, const ScopedKey& key, const uint8_t* iv8, uint8_t* buf, uint64_t n, uint64_t offset) {
  const size_t nd = ctx->devs.size();
  if (nd == 1) { aes_ctr_host_range(ctx->devs[0], key, iv8, buf, n, offset); return; }
  std::vector<std::string> errs(nd);
  std::vector<int> codes(nd, 0);
  std::vector<std::thread> th;
  for (size_t k = 0; k < nd; ++k) {
    const uint64_t lo = (uint64_t)((unsigned __int128)n * k / nd), hi = (uint64_t)((unsigned __int128)n * (k + 1) / nd);
    th.emplace_back([&, k, lo, hi]() {
      try { aes_ctr_host_range(ctx->devs[k], key, iv8, buf + lo, hi - lo, offset + lo); }
      catch (const Failure& f) { codes[k] = f.code; errs[k] = f.what(); }
      catch (const std::exception& e) { codes[k] = ZPQ_E_CUDA; errs[k] = e.what(); }
    });
  }
  for (auto& t : th) t.join();
  for (size_t k = 0; k < nd; ++k) if (codes[k]) throw Failure(codes[k], errs[k]);
}

}  // namespace

// =========================================================================================
extern "C" {

const char* zpq_version(void) { return "zpaqb200 0.1 sm_100a"; }

int zpq_create(const int* device_ids, int ndev, zpq_ctx** out) {
  if (!out) return ZPQ_E_ARG;
  *out = nullptr;
  std::unique_ptr<zpq_ctx> ctx(new zpq_ctx);
  int rc = guarded(nullptr, [&]() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1)
      throw Failure(ZPQ_E_CUDA, std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    std::vector<int> ids;
    if (ndev <= 0) { int cur = 0; CU(cudaGetDevice(&cur)); ids.push_back(cur); }
    else for (int i = 0; i < ndev; ++i) ids.push_back(device_ids ? device_ids[i] : i);
    for (int id : ids) if (id < 0 || id >= count) throw Failure(ZPQ_E_ARG, "device id out of range");
    ctx->devs.resize(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) ctx->devs[i].init(ids[i]);
  });
  if (rc != ZPQ_OK) { for (auto& d : ctx->devs) d.fini(); return rc; }
  *out = ctx.release();
  return ZPQ_OK;
}

void zpq_destroy(zpq_ctx* ctx) {
  if (!ctx) return;
  for (auto& d : ctx->devs) d.fini();
  delete ctx;
}

const char* zpq_last_error(zpq_ctx* ctx) {
  if (ctx) return ctx->err.c_str();
  std::lock_guard<std::mutex> g(g_create_mutex);
  return g_create_error.c_str();
}

int zpq_set_stream(zpq_ctx* ctx, void* cuda_stream) {
  if (!ctx) return ZPQ_E_ARG;
  Device& d = ctx->devs[0];
  d.stream = cuda_stream ? (cudaStream_t)cuda_stream : d.own;
  return ZPQ_OK;
}

int zpq_set_max_resident(zpq_ctx* ctx, uint32_t max_blocks) {
  if (!ctx) return ZPQ_E_ARG;
  ctx->max_resident = max_blocks;
  return ZPQ_OK;
}

int64_t zpq_make_config(const char* method, int* args9, char* text, uint64_t text_cap) {
  if (!method || !args9) return ZPQ_E_ARG;
  std::string r;
  int rc = guarded(nullptr, [&]() { r = make_config(method, args9); });
  return rc ? rc : copy_out(r, text, text_cap);
}

int64_t zpq_expand_method(const char* method, const uint8_t* block, uint64_t n, char* out, uint64_t cap) {
  if (!method || (!block && n)) return ZPQ_E_ARG;
  std::string r;
  int rc = guarded(nullptr, [&]() { r = expand_method(method, block, n); });
  return rc ? rc : copy_out(r, out, cap);
}

int zpq_compile_config(const char* config, const int* args9, uint8_t* hdr, uint64_t hdr_cap, uint64_t* hdr_len,
                       uint8_t* pcomp, uint64_t pcomp_cap, uint64_t* pcomp_len) {
  if (!config || !hdr_len || !pcomp_len) return ZPQ_E_ARG;
  return guarded(nullptr, [&]() {
    Bytes h, p;
    compile_config(config, args9, h, p, nullptr);
    *hdr_len = h.size(); *pcomp_len = p.size();
    if (h.size() > hdr_cap || p.size() > pcomp_cap) throw Failure(ZPQ_E_OUTPUT, "buffer too small");
    if (hdr) memcpy(hdr, h.data(), h.size());
    if (pcomp && !p.empty()) memcpy(pcomp, p.data(), p.size());
  });
}

int64_t zpq_builtin_model(int level, uint8_t* hdr, uint64_t hdr_cap) {
  Bytes h;
  int rc = guarded(nullptr, [&]() { builtin_model(level, h); });
  if (rc) return rc;
  if (hdr) { if (h.size() > hdr_cap) return ZPQ_E_OUTPUT; memcpy(hdr, h.data(), h.size()); }
  return (int64_t)h.size();
}

double zpq_block_memory(const uint8_t* hdr, uint64_t hdr_len) {
  double v = -1;
  guarded(nullptr, [&]() { Header h; parse_header(hdr, hdr_len, h); v = header_memory(h); });
  return v;
}

int64_t zpq_device_state_bytes(const uint8_t* hdr, uint64_t hdr_len, int for_decode) {
  int64_t v = -1;
  int rc = guarded(nullptr, [&]() {
    Header h; parse_header(hdr, hdr_len, h);
    std::unique_ptr<Plan> p(new Plan);
    build_plan(h, for_decode != 0, 48 * 1024, *p);
    v = (int64_t)p->arena_bytes;
  });
  return rc ? rc : v;
}

int64_t zpq_device_state_bytes_for(const uint8_t* hdr, uint64_t hdr_len, int for_decode, uint64_t max_block_bytes) {
  int64_t v = -1;
  int rc = guarded(nullptr, [&]() {
    Header h; parse_header(hdr, hdr_len, h);
    std::unique_ptr<Plan> p(new Plan);
    // the stream bound the schedulers use: compress_on_device (transformed block + preamble), decompress_range (raw slot)
    const uint64_t bound = for_decode ? max_block_bytes + 16 + (max_block_bytes + 16) / 8 + 70000 : max_block_bytes + max_block_bytes / 16 + 65536 + 3 + 64;
    build_plan(h, for_decode != 0, 48 * 1024, *p, 0, false, max_block_bytes ? bound : 0);
    v = (int64_t)p->arena_bytes;
  });
  return rc ? rc : v;
}

int zpq_encoder_plan(const uint8_t* hdr, uint64_t hdr_len, uint32_t smem_bytes, uint32_t blocks_per_sm, int32_t* out8) {
  if (!hdr || !out8) return ZPQ_E_ARG;
  return guarded(nullptr, [&]() {
    Header h; parse_header(hdr, hdr_len, h);
    for (int i = 0; i < 8; ++i) out8[i] = 0;
    if (h.n < 1 || h.n > 32) return;
    const uint32_t G = h.n <= 8 ? 8u : h.n <= 16 ? 16u : 32u, B = 32 / G;
    std::unique_ptr<Plan> p(new Plan);
    build_plan(h, false, 48 * 1024, *p, (int)G);
    const uint32_t roles = p->duo_split ? 4u : 3u;
    uint32_t wb = std::min(std::max(blocks_per_sm, 1u), std::min((15u / roles) * B, 32u));
    bool ok = false;
    for (; wb >= 1 && !ok; --wb) {
      SmemLayout L;
      const uint32_t common = common_smem(*p, L);
      const uint32_t avail = smem_bytes > common ? smem_bytes - common : 0;
      build_plan(h, false, (avail / wb) & ~127u, *p, (int)G);
      ok = p->duo_ok && p->pipe_maps && (uint64_t)wb * p->smem_warp_bytes <= avail;
      if (ok) break;
    }
    out8[0] = ok ? 1 : 0; out8[1] = (int32_t)G; out8[2] = (int32_t)roles; out8[3] = ok ? (int32_t)wb : 0;
    out8[4] = (int32_t)p->smem_warp_bytes; out8[5] = p->coder_delay; out8[6] = p->duo_split;
    out8[7] = ok ? (int32_t)(1 + roles * ((wb + B - 1) / B)) : 0;
  });
}

int zpq_compress_blocks_model(zpq_ctx* ctx, const uint8_t* hdr, uint64_t hdr_len, const uint8_t* pcomp, uint64_t pcomp_len,
                              const int* args9, const uint8_t* in, const uint64_t* in_off, uint32_t nb,
                              const char* filename0, const char* comment0, int dosha1, int with_tag, uint8_t* out,
                              uint64_t out_cap, uint64_t* out_off) {
  if (!ctx || !in_off || !out_off || (!in && nb && in_off[nb] > in_off[0]) || !out) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    out_off[0] = 0;
    if (!nb) return;
    Model M;
    model_from_header_bytes(hdr, hdr_len, pcomp, pcomp_len, args9, M);
    std::vector<std::string> fn(1, filename0 ? filename0 : ""), cm(1, comment0 ? comment0 : "");
    compress_model(ctx, M, in, in_off, 0, nb, fn, cm, dosha1 != 0, with_tag != 0, out, out_cap, 0, out_off);
  });
}

int zpq_compress_blocks_level(zpq_ctx* ctx, int level, const uint8_t* in, const uint64_t* in_off, uint32_t nb,
                              const char* filename0, const char* comment0, int dosha1, int with_tag, uint8_t* out,
                              uint64_t out_cap, uint64_t* out_off) {
  if (!ctx) return ZPQ_E_ARG;
  Bytes h;
  int rc = guarded(ctx, [&]() { builtin_model(level, h); });
  if (rc) return rc;
  return zpq_compress_blocks_model(ctx, h.data(), h.size(), nullptr, 0, nullptr, in, in_off, nb, filename0, comment0, dosha1,
                                   with_tag, out, out_cap, out_off);
}

int zpq_compress_blocks(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, const char* method,
                        const char* filename0, const char* comment0, int dosha1, uint8_t* out, uint64_t out_cap,
                        uint64_t* out_off) {
  if (!ctx || !in_off || !out_off || !method || !out || (!in && nb && in_off[nb] > in_off[0])) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    out_off[0] = 0;
    // derive each block's model (LibZPAQ.cs:128-300); consecutive blocks with identical models
    // form one device batch
    uint32_t i = 0;
    uint64_t base = 0;
    // levels 5..9 choose their periodic models from the block's byte-gap histogram (LibZPAQ.cs:242-280): counted on the device
    std::vector<int> gaps;
    const bool analyse = method_needs_analysis(method);
    if (analyse) device_gap_histograms(ctx, in, in_off, nb, gaps);
    // derive each block's model (LibZPAQ.cs:128-300)
    std::vector<Model> models(nb);
    for (uint32_t b = 0; b < nb; ++b) {
      Model& M = models[b];
      const uint64_t n = in_off[b + 1] - in_off[b];
      std::string x = expand_method_gaps(method, n, analyse ? gaps.data() + (size_t)b * kGapBins : nullptr);
      std::string cfg = make_config(x, M.args);
      Bytes h;
      compile_config(cfg, M.args, h, M.pcomp, nullptr);
      parse_header(h.data(), h.size(), M.hdr);
    }
    auto same_model = [&](uint32_t a, uint32_t b) {
      return models[a].hdr.wire == models[b].hdr.wire && models[a].pcomp == models[b].pcomp && memcmp(models[a].args, models[b].args, sizeof(models[a].args)) == 0;
    };
    auto names = [&](uint32_t b, std::vector<std::string>& fn, std::vector<std::string>& cm) {
      const uint64_t n = in_off[b + 1] - in_off[b];
      fn.push_back(b == 0 && filename0 ? filename0 : "");
      std::string c = std::to_string(n);                       // LibZPAQ.cs:298-299
      if (b == 0 && comment0 && *comment0) c += std::string(" ") + comment0;
      cm.push_back(c);
    };
    // blocks of one model form one device batch: runs of consecutive blocks where that is all there is ...
    uint32_t runs = 0;
    std::vector<uint32_t> rep;                                  // first block of every distinct model
    std::vector<uint32_t> cls(nb, 0);
    for (uint32_t b = 0; b < nb; ++b) {
      if (b == 0 || !same_model(b, b - 1)) ++runs;
      uint32_t k = 0;
      while (k < rep.size() && !same_model(rep[k], b)) ++k;
      if (k == rep.size()) rep.push_back(b);
      cls[b] = k;
    }
    if (runs == rep.size()) {
      while (i < nb) {
        uint32_t j = i + 1;
        while (j < nb && same_model(i, j)) ++j;
        std::vector<std::string> fn, cm;
        for (uint32_t b = i; b < j; ++b) names(b, fn, cm);
        compress_model(ctx, models[i], in, in_off, i, j - i, fn, cm, dosha1 != 0, true, out, out_cap, base, out_off);
        base = out_off[j];
        i = j;
      }
      return;
    }
    // ... and otherwise (data-dependent models of levels 5..9, ragged block sizes: the same model comes back after other
    // models) all blocks of a model, gathered on the host, so that a batch is as large as it can be; the archive blocks go
    // back into block order
    std::vector<Bytes> arcs(nb);
    for (uint32_t k = 0; k < rep.size(); ++k) {
      std::vector<uint32_t> ids;
      for (uint32_t b = 0; b < nb; ++b) if (cls[b] == k) ids.push_back(b);
      Bytes gin;
      std::vector<uint64_t> goff(ids.size() + 1, 0);
      std::vector<std::string> fn, cm;
      for (size_t t = 0; t < ids.size(); ++t) {
        const uint32_t bb = ids[t];
        gin.insert(gin.end(), in + in_off[bb], in + in_off[bb + 1]);
        goff[t + 1] = gin.size();
        names(bb, fn, cm);
      }
      gin.resize(gin.size() + 64);
      Bytes gout(gin.size() + gin.size() / 4 + (models[rep[k]].hdr.wire.size() + models[rep[k]].pcomp.size() * 4 + 70000) * ids.size());
      std::vector<uint64_t> gooff(ids.size() + 1, 0);
      compress_model(ctx, models[rep[k]], gin.data(), goff.data(), 0, (uint32_t)ids.size(), fn, cm, dosha1 != 0, true, gout.data(), gout.size(), 0, gooff.data());
      for (size_t t = 0; t < ids.size(); ++t) arcs[ids[t]].assign(gout.begin() + gooff[t], gout.begin() + gooff[t + 1]);
    }
    for (uint32_t b = 0; b < nb; ++b) {
      if (base + arcs[b].size() > out_cap) throw Failure(ZPQ_E_OUTPUT, "output buffer too small");
      memcpy(out + base, arcs[b].data(), arcs[b].size());
      base += arcs[b].size();
      out_off[b + 1] = base;
    }
  });
}

int zpq_compress_blocks_model_dev(zpq_ctx* ctx, const uint8_t* hdr, uint64_t hdr_len, const uint8_t* pcomp, uint64_t pcomp_len,
                                  const int* args9, const uint8_t* d_in, const uint64_t* h_in_off, uint32_t nb, int dosha1,
                                  int with_tag, uint8_t* d_out, uint64_t out_cap, uint64_t* h_out_off) {
  if (!ctx || !d_in || !h_in_off || !d_out || !h_out_off) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    h_out_off[0] = 0;
    if (!nb) return;
    Model M;
    model_from_header_bytes(hdr, hdr_len, pcomp, pcomp_len, args9, M);
    CompressTask T;
    T.model = &M; T.d_in_ext = d_in; T.in_off = h_in_off; T.first = 0; T.count = nb;
    T.dosha1 = dosha1 != 0; T.with_tag = with_tag != 0; T.d_out_ext = d_out; T.d_out_cap = out_cap;
    compress_on_device(ctx, ctx->devs[0], T, nullptr, 0);
    for (uint32_t i = 0; i <= nb; ++i) h_out_off[i] = T.frame_off[i];
  });
}

int64_t zpq_find_blocks(const uint8_t* archive, uint64_t n, uint64_t* offsets, uint64_t max_blocks) {
  int64_t r = 0;
  int rc = guarded(nullptr, [&]() { r = find_blocks(archive, n, offsets, max_blocks); });
  return rc ? rc : r;
}

int64_t zpq_decompressed_bound(const uint8_t* in, const uint64_t* in_off, uint32_t nb) {
  int64_t total = 0;
  int rc = guarded(nullptr, [&]() {
    for (uint32_t i = 0; i < nb; ++i) {
      BlockRef b;
      parse_block(in + in_off[i], in_off[i + 1] - in_off[i], b);
      for (const SegmentRef& s : b.segs) total += s.size_hint >= 0 ? s.size_hint : (int64_t)(s.data_len * 64 + 65536);
      total += 16;
    }
  });
  return rc ? rc : total;
}

int zpq_decompress_blocks(zpq_ctx* ctx, const uint8_t* in, const uint64_t* in_off, uint32_t nb, uint8_t* out, uint64_t out_cap,
                          uint64_t* out_off, uint8_t* sha1_status, uint8_t* block_status) {
  if (!ctx || !in || !in_off || !out_off || (!out && out_cap)) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    out_off[0] = 0;
    if (!nb) return;
    decompress_all(ctx, in, in_off, nb, out, out_cap, out_off, sha1_status, block_status);
  });
}

int64_t zpq_specialize_model(const uint8_t* hdr, uint64_t hdr_len, char* source, uint64_t source_cap, char* log, uint64_t log_cap) {
  int64_t size = -1;
  std::string src, msg;
  try {
    Header h;
    parse_header(hdr, hdr_len, h);
    bool compiled = false;
    src = generate_model_source(h, "Model_rt", "zpq_enc_rt", "zpq_dec_rt", &compiled, nullptr, nullptr);
    Bytes cubin = nvrtc_compile(src);
    size = (int64_t)cubin.size();
    msg = compiled ? "HCOMP compiled" : "HCOMP interpreted";
  } catch (const Failure& f) { msg = f.what(); size = f.code; }
  catch (const std::exception& e) { msg = e.what(); size = ZPQ_E_CONFIG; }
  copy_out(src, source, source_cap);
  copy_out(msg, log, log_cap);
  return size;
}

int64_t zpq_post_kind(int ph, int pm, const uint8_t* pcomp, uint64_t len) {
  try {
    std::vector<PostCandidate> cands;
    post_candidates(ph, pm, cands);
    for (const PostCandidate& c : cands) {
      if (c.prog.size() != len) continue;
      bool same = true;
      for (uint64_t i = 0; i < len && same; ++i) same = (int64_t)i == c.wild || pcomp[i] == c.prog[i];
      if (same) return (int64_t)(c.kind | c.e8 << 4 | (c.wild >= 0 ? (uint32_t)pcomp[c.wild] : c.param) << 8);
    }
    return 0;
  } catch (const Failure& f) { return f.code; }
}

int64_t zpq_specialize_pcomp(int ph, int pm, const uint8_t* pcomp, uint64_t len, char* source, uint64_t source_cap, char* log, uint64_t log_cap) {
  if (!pcomp || !len) return ZPQ_E_ARG;
  std::string src, lg;
  const int64_t n = post_program_cubin(Bytes(pcomp, pcomp + len), ph, pm, &src, &lg);
  copy_out(src, source, source_cap);
  copy_out(lg, log, log_cap);
  return n;
}

int zpq_get_stats(zpq_ctx* ctx, zpq_stats* out) {
  if (!ctx || !out) return ZPQ_E_ARG;
  *out = ctx->devs[0].stats;
  return ZPQ_OK;
}

int zpq_scrypt(const uint8_t* pw, uint64_t pwlen, const uint8_t* salt, uint64_t saltlen, uint64_t n, uint32_t r, uint32_t p,
               uint8_t* out, uint64_t outlen) {
  if ((!pw && pwlen) || (!salt && saltlen) || (!out && outlen)) return ZPQ_E_ARG;
  return guarded(nullptr, [&]() { scrypt(pw, pwlen, salt, saltlen, n, r, p, out, outlen); });
}

int zpq_stretch_key(const uint8_t* in32, const uint8_t* salt32, uint8_t* out32) {
  if (!in32 || !salt32 || !out32) return ZPQ_E_ARG;
  return guarded(nullptr, [&]() { scrypt(in32, 32, salt32, 32, 16384, 8, 1, out32, 32); });
}

int zpq_aes_ctr(zpq_ctx* ctx, const uint8_t* key, int keylen, const uint8_t* iv8, uint8_t* buf, uint64_t n, uint64_t offset) {
  if (!ctx) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    check_aes_range(buf, n, offset);
    const ScopedKey k(key, keylen);
    aes_ctr_host(ctx, k, iv8, buf, n, offset);
  });
}

int zpq_aes_ctr_dev(zpq_ctx* ctx, const uint8_t* key, int keylen, const uint8_t* iv8, uint8_t* d_buf, uint64_t n, uint64_t offset) {
  if (!ctx) return ZPQ_E_ARG;
  return guarded(ctx, [&]() {
    check_aes_range(d_buf, n, offset);
    const ScopedKey k(key, keylen);
    Device& d = ctx->devs[0];
    CU(cudaSetDevice(d.id));
    cudaStream_t s = d.stream;
    d.stats = zpq_stats{};
    snprintf(d.stats.kernel, sizeof d.stats.kernel, "%s", k.name().c_str());
    if (!n) return;
    d.t_all.start(s);
    d.t_kern.start(s);
    CU(launch_aes_ctr(k.k, iv8, d_buf, n, offset, s));
    d.t_kern.stop(s);
    d.t_all.stop(s);
    CU(cudaStreamSynchronize(s));
    d.stats.kernel_ms = d.t_kern.ms(); d.stats.total_ms = d.t_all.ms(); d.stats.launches = 1;
  });
}

}  // extern "C"
