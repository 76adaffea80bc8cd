#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native ZPAQ block codec.

Metric (BASELINE.json): compress & decompress MB/s (MB = 10^6 input bytes), method-2 (mid.cfg =
Compressor.startBlock(2), SURVEY.md 8d C2a), 1 MB blocks (1,044,480 B), byte-exact, 1/2/4/8 B200.

A "step" is one pass of the compress hot path over one batch of synthetic mixed text/binary blocks
(the batch is as many blocks as fit resident on one GPU: one warp per block, ~106 MiB of model
state per block).  Blocks are independent, so N GPUs = N ranks each coding its own batch (weak
scaling, no collective on the data path; NCCL is used for the barrier and the max-over-ranks only).

  value     compress MB/s, whole job, inputs and outputs resident in HBM (kernel path only)
  e2e       the same through the public C ABI with HOST buffers: pinned H2D of every block and
            D2H of every archive inside the timed region
  roofline  HBM roofline of the coding kernel from the algorithmic bytes of SURVEY.md 8d
  cpu_baseline / --impl reference
            the CPU oracle (a C++ restatement of the reference; ZPAQSharp itself cannot be built,
            SURVEY.md 8c) timed on the box's host cores on a bounded sample of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = (0x100000 << 0) - 4096          # 1,044,480 B  (LibZPAQ.cs:94)
BLOCK_4MB = (0x100000 << 2) - 4096      # 4,190,208 B
BLOCK_16MB = (0x100000 << 4) - 4096     # 16,773,120 B
TOTAL_BLOCKS = 8192                     # the 8 GB stream of BASELINE.json configs[1]
LEVEL = 2                               # mid.cfg
ALGO_BYTES_PER_INPUT_BYTE = 950.0       # SURVEY.md 8d: A(C2a), state read+write at the reference's granularity
METRIC = "compress MB/s, method-2 (mid.cfg) 1 MB blocks, byte-exact"


def lz_method(a0):  return "x%d,1,4,0,7,%d,1" % (a0, 21 + a0)                   # what method "20" expands to (LibZPAQ.cs:189-198)
def lzcm_method(a0): return "x%d,2,12,0,7,%d,1c0,0,511i2m" % (a0, 21 + a0)       # level-3 default + mixer (SURVEY 8d C2c)
def bwt_method(a0): return "x%d,3ci1" % a0                                       # what "3N,128,1" expands to on text (LibZPAQ.cs:207-208)


# SURVEY.md 8d: the BASELINE.json configs restated.  how = ("level", n) -> Compressor.startBlock(n); ("method", s) -> compressBlock(s).
# max_blocks bounds the batch of the non-headline configs so that the default run stays within minutes.
CONFIGS = {
    "C1": {"what": "configs[0]: single order-2 CM, method x0,0c256,0,255,255, 1,044,480-byte blocks of synthetic text",
           "kind": "text", "block": BLOCK, "how": ("method", "x0,0c256,0,255,255"), "max_blocks": 2960,
           "metric": "compress MB/s, order-2 CM 1 MB blocks, byte-exact"},
    "C2a": {"what": "BASELINE configs[1]: mid.cfg (Compressor.startBlock(2)), 1,044,480-byte blocks of the 8192-block (8 GB) synthetic mixed text/binary stream",
            "kind": "mixed", "block": BLOCK, "how": ("level", 2), "max_blocks": 148 * 16, "metric": METRIC},
    "C2b": {"what": "configs[1] read literally: libzpaq method 20 = x0,1,4,0,7,21,1 (bit-packed LZ77, suffix-array matcher, stored), 1 MB mixed blocks",
            "kind": "mixed", "block": BLOCK, "how": ("method", lz_method(0)), "max_blocks": 1776,
            "metric": "compress MB/s, method 20 (LZ77 stored) 1 MB blocks, byte-exact"},
    "C2c": {"what": "configs[1]'s parenthesis: x0,2,12,0,7,21,1c0,0,511i2m (byte LZ77 + ICM/ISSE chain + MIX), 1 MB mixed blocks",
            "kind": "mixed", "block": BLOCK, "how": ("method", lzcm_method(0)), "max_blocks": 1776,
            "metric": "compress MB/s, LZ77+ICM/ISSE+MIX 1 MB blocks, byte-exact"},
    "C3": {"what": "configs[2]: method 32,128,1 = x2,3ci1 (BWT + ICM/ISSE), 4,190,208-byte blocks of synthetic text",
           "kind": "text", "block": BLOCK_4MB, "how": ("method", bwt_method(2)), "max_blocks": 592,
           "metric": "compress MB/s, method 3 (BWT) 4 MB blocks, byte-exact"},
    "C4": {"what": "configs[3]: max.cfg (Compressor.startBlock(3), 22 components: CONST/ICM/ISSE chain/MATCH/MIX/MIX2/SSE with a word-model HCOMP), 1 MB mixed blocks",
           "kind": "mixed", "block": BLOCK, "how": ("level", 3), "max_blocks": 740,
           "metric": "compress MB/s, max.cfg 1 MB blocks, byte-exact"},
}


def shard_blocks(total: int, rank: int, world: int):
    """Contiguous block range of `rank` (blocks are independent: SURVEY.md 8e)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_max_time(t: float, device: str) -> float:
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return t
    x = torch.tensor([t], dtype=torch.float64, device=device)
    dist.all_reduce(x, op=dist.ReduceOp.MAX)
    return float(x.item())


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _reference_block_coder():
    """The reference's own text for the hot loop, when oracle/_ref holds it: Predictor.init / predict0 / update0 / find,
    ZPAQL.execute and Encoder.encode compiled by oracle/build_ref.py (prebuilt; nothing is read from /root/reference at
    run time).  Returns code(block) -> coded bytes of the block, or None."""
    import ctypes as C
    import hashlib
    try:
        from oracle import build_ref, frontend
        path = build_ref.build_predictor()
        if not path or not os.path.exists(path):
            return None
        L = C.CDLL(path)
        kat = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_kat.json")))
        tabs = [np.asarray(kat["sdt2k"], dtype=np.int32), np.asarray(kat["sdt"], dtype=np.int32), np.asarray(kat["ssquasht"], dtype=np.uint16),
                np.asarray(kat["stdt"], dtype=np.int32), np.asarray(kat["sns"], dtype=np.uint8)]
        L.ref_predictor_tables.argtypes = [C.c_void_p] * 5
        L.ref_predictor_tables(*[t.ctypes.data for t in tabs])
        L.ref_code_block.argtypes = [C.c_char_p, C.c_ulonglong, C.c_char_p, C.c_ulonglong, C.c_char_p, C.c_ulonglong, C.c_void_p, C.c_ulonglong]
        L.ref_code_block.restype = C.c_longlong
        hdr = bytes(frontend.builtin_model(LEVEL)[0])
    except Exception:
        return None

    def code(b):
        hashlib.sha1(b).digest()                    # compressBlock hashes the block first (LibZPAQ.cs:143-155; the SHA1 class itself is missing)
        cap = len(b) + len(b) // 4 + 4096
        out = C.create_string_buffer(cap)
        n = L.ref_code_block(hdr, len(hdr), b"\x00", 1, b, len(b), out, cap)      # ctypes releases the GIL: one block per thread
        if n < 0:
            raise RuntimeError("reference coder failed")
        return out.raw[:n]
    return code


def _reference_block_codec(level: int = LEVEL):
    """The reference's own text for the WHOLE block path, when oracle/_ref holds it: Compressor.writeTag / startBlock(level) /
    startSegment / postProcess / compress / endSegment / endBlock over Encoder, Predictor and ZPAQL text, and the way back
    through Decompresser / Decoder / PostProcessor (oracle/build_ref.py; prebuilt, nothing is read from /root/reference at
    run time).  Returns (compress(block) -> archive block, decompress(archive, n) -> bytes) or None."""
    import ctypes as C
    import hashlib
    try:
        from oracle import build_ref
        pc, pd = build_ref.build_compressor(), build_ref.build_decompresser()
        if not pc or not pd or not os.path.exists(pc) or not os.path.exists(pd):
            return None
        kat = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_kat.json")))
        tabs = [np.asarray(kat["sdt2k"], dtype=np.int32), np.asarray(kat["sdt"], dtype=np.int32), np.asarray(kat["ssquasht"], dtype=np.uint16),
                np.asarray(kat["stdt"], dtype=np.int32), np.asarray(kat["sns"], dtype=np.uint8)]
        Lc, Ld = C.CDLL(pc), C.CDLL(pd)
        for L in (Lc, Ld):
            L.ref_predictor_tables.argtypes = [C.c_void_p] * 5
            L.ref_predictor_tables(*[t.ctypes.data for t in tabs])
        Lc.ref_compress_block.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_ulonglong,
                                          C.c_char_p, C.c_int, C.c_void_p, C.c_ulonglong]
        Lc.ref_compress_block.restype = C.c_longlong
        Ld.ref_decompress.argtypes = [C.c_char_p, C.c_ulonglong, C.c_void_p, C.c_ulonglong, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        Ld.ref_decompress.restype = C.c_longlong
    except Exception:
        return None

    def comp(b):
        sha = hashlib.sha1(b).digest()              # compressBlock hashes the block first (LibZPAQ.cs:143-155; the SHA1 class itself is missing)
        cap = len(b) + len(b) // 4 + 4096
        out = C.create_string_buffer(cap)
        n = Lc.ref_compress_block(level, None, None, 0, None, str(len(b)).encode(), b, len(b), sha, 1, out, cap)   # ctypes releases the GIL
        if n < 0 or n > cap:
            raise RuntimeError("reference Compressor text failed")
        return out.raw[:n]

    def decomp(a, n):
        out = C.create_string_buffer(n + 64)
        marks = C.create_string_buffer(21 * 4)
        nseg = C.c_int(0)
        m = Ld.ref_decompress(a, len(a), out, n + 64, marks, 4, C.byref(nseg))
        if m < 0:
            raise RuntimeError("reference Decompresser text failed")
        return out.raw[:m]
    return comp, decomp


COMP_LEN = [0, 2, 3, 2, 3, 4, 6, 6, 3, 5]        # Component.cs:27-43


def algorithmic_bytes(hdr: bytes, state_bytes: int, block_bytes: int, ratio: float, preproc: int) -> float:
    """SURVEY.md 8d: A(config), bytes of state traffic per input byte at the reference's own granularity (read + write-back),
    plus stream I/O, amortised table initialisation and, for LZ77 / BWT pre-processing, the suffix-array floor."""
    a = 1.0 + ratio
    i = 7
    for _ in range(hdr[6]):
        t = hdr[i]
        a += {2: 64, 3: 64, 8: 64, 4: 10, 6: 32, 9: 96}.get(t, 0)
        if t == 7:
            a += 64 * hdr[i + 3]
        i += COMP_LEN[t]
    a += state_bytes / max(block_bytes, 1)
    if preproc:
        a += 9.0                                  # 4 B SA write + 4 B SA read + 1 B transformed stream
    return a


def model_of(cfg):
    """(header bytes, pcomp bytes, args[9]) of a config, through the library's own front end."""
    from zpaqsharp_b200 import libzpaq as z
    how, arg = cfg["how"]
    if how == "level":
        return z.builtin_model(arg), b"", [0] * 9
    text, args = z.make_config(arg)
    hdr, pcomp = z.compile_config(text, args)
    return hdr, pcomp, list(args)


def host_info():
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


def cpu_baseline(cfg_id: str = "C2a", seconds_budget: float = 20.0, decompress: bool = True, max_threads: int | None = None):
    """Time the CPU path (one block per host thread) on a bounded sample of the workload: the reference's own text when
    oracle/_ref holds it and the config is a built-in level (kind "reference": the whole Compressor / Decompresser path), else
    the oracle port (kind "port")."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po
    from tools import synth
    po.build()
    cfg = CONFIGS[cfg_id]
    how, arg = cfg["how"]
    bs = cfg["block"]
    cores = os.cpu_count() or 1
    nthr = min(cores, max_threads or cores)
    data = synth.blocks(cfg["kind"], 0, nthr, bs)
    blocks = [data[i * bs:(i + 1) * bs].tobytes() for i in range(nthr)]
    codec = _reference_block_codec(arg) if how == "level" else None

    def comp(b):
        return po.compress_block_level(b, arg) if how == "level" else po.compress_block(b, arg)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(nthr) as ex:
        arcs = list(ex.map(comp, blocks))
    t_port = time.perf_counter() - t0
    out = {"value": nthr * bs / 1e6 / t_port, "unit": "MB/s", "cores": nthr, "kind": "port",
           "sample": "%d blocks of %d B (one per host thread), %s, oracle C++ -O2" % (nthr, bs, cfg_id),
           "seconds": t_port}
    out.update(host_info())
    if codec is not None:
        t0 = time.perf_counter()
        with ThreadPoolExecutor(nthr) as ex:
            rarcs = list(ex.map(codec[0], blocks))
        t_ref = time.perf_counter() - t0
        assert rarcs == arcs, "reference text and oracle disagree"          # whole archive blocks, byte for byte
        out.update({"value": nthr * bs / 1e6 / t_ref, "kind": "reference", "seconds": t_ref, "port_value": nthr * bs / 1e6 / t_port,
                    "sample": "%d blocks of %d B (one per host thread), %s; the reference's own Compressor.startBlock(%d) .. endBlock "
                              "path (Compressor, Encoder, Predictor.init/predict0/update0/find, ZPAQL text compiled -O2 from "
                              "/root/reference by oracle/build_ref.py, + SHA-1 of the block); archive blocks checked byte for byte "
                              "against the oracle's" % (nthr, bs, cfg_id, arg)})
    if decompress and out["seconds"] < seconds_budget:
        dec = (lambda a: codec[1](a, bs)) if codec else (lambda a: po.decompress(a, cap=bs + 64)[0])
        t0 = time.perf_counter()
        with ThreadPoolExecutor(nthr) as ex:
            back = list(ex.map(dec, arcs))
        t_d = time.perf_counter() - t0
        assert all(b == s for b, s in zip(back, blocks))
        out["decompress_value"] = nthr * bs / 1e6 / t_d        # the reference's Decompresser text when present, else the oracle port
        out["decompress_kind"] = "reference" if codec else "port"
    if cfg_id == "C2a":
        t0 = time.perf_counter()
        (codec[0] if codec else comp)(blocks[0])
        out["single_core_value"] = bs / 1e6 / (time.perf_counter() - t0)
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores, rank 0 only: the reference's own
    text compiled into oracle/_ref (kind "reference"), or the oracle port when that is missing / for method-string configs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg_id = args.config if args.config in CONFIGS else "C2a"
    cfg = workload_config(cfg_id, args.batch_blocks or None, args.gpus)
    vals = []
    for _ in range(args.warmup):
        cpu_baseline(cfg_id, decompress=False)
    t_steps = []
    base = None
    for _ in range(max(1, args.steps)):
        t0 = time.perf_counter()
        base = cpu_baseline(cfg_id, decompress=False)
        t_steps.append(time.perf_counter() - t0)
        vals.append(base["value"])
    v = sum(vals) / len(vals)
    base["value"] = v
    dec = cpu_baseline(cfg_id, decompress=True)
    _emit({
        "impl": "reference", "metric": CONFIGS[cfg_id]["metric"], "value": v, "unit": "MB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(t_steps) / len(t_steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": cfg, "cpu_baseline": base,
        "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "decompress": {"e2e_value": dec.get("decompress_value"), "unit": "MB/s", "kind": dec.get("decompress_kind")},
        "note": "kind reference: Compressor/Encoder/Predictor/ZPAQL text of the reference compiled from /root/reference (oracle/build_ref.py); "
                "kind port: the C++ oracle restating it (ZPAQSharp as a whole is not buildable)",
    })


def wave_blocks(cfg_id: str, n_gpus_unused: int = 1) -> int:
    """Blocks of one resident wave on a 180 GB B200 (what bench.py codes per GPU and step; deterministic so that the reference
    arm, which has no GPU to ask, names the same config)."""
    return {"C2a": 1776, "C4": 740}.get(cfg_id, CONFIGS[cfg_id]["max_blocks"])


def workload_config(cfg_id, batch_blocks, n_gpus):
    cfg = CONFIGS[cfg_id]
    return {"workload": cfg["what"], "config_id": cfg_id,
            "block_bytes": cfg["block"], "stream_blocks": TOTAL_BLOCKS, "batch_blocks_per_gpu": batch_blocks or wave_blocks(cfg_id),
            "parallelism": "blocks x%d GPUs, no collective" % n_gpus,
            "l2_policy": "inputs larger than L2 (batch >= 1 GB per GPU, per-block model state in HBM)",
            "sha1": True}


# ------------------------------------------------------------------------------------------------------------------
class Rig:
    """What every measurement needs: the library context on this rank's GPU, torch's stream, the rank geometry."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from zpaqsharp_b200 import libzpaq as z
        self.torch, self.dist, self.z = torch, dist, z
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dev = "cuda:%d" % self.local
        self.host_group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device(self.dev))
            self.host_group = dist.new_group(backend="gloo")     # host-side waits that must not occupy an SM
        self.open()

    def open(self):
        self.ctx = self.z.Context([self.local])
        self.stream = self.torch.cuda.Stream(device=self.dev)       # the library launches on this stream; events are recorded on it
        self.torch.cuda.set_stream(self.stream)
        self.ctx.set_stream(self.stream.cuda_stream)

    def close(self):
        self.ctx.close()
        self.torch.cuda.synchronize()
        self.torch.cuda.empty_cache()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_time(self, t):
        return reduce_max_time(t, self.dev)


DUMP_POOL = 148          # blocks the dump samples from: one per SM, fewer than any default batch holds, so the dump does not
                         # depend on the batch size the free device memory allows
DUMP_SAMPLE = 16         # archive blocks stored byte for byte
DUMP_SEED = 20261020
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, d_out, ooff: np.ndarray, B: int):
    """What the device-resident compress returned in its last step, as float arrays for comparing two builds: the archive size
    of each of the first min(B, DUMP_POOL) blocks and the archive bytes of a fixed, seeded sample of them (with their indices).
    Blocks are coded independently, so these do not depend on how many blocks the batch holds beyond the pool."""
    pool = min(B, DUMP_POOL)
    sizes = np.diff(ooff[:pool + 1].astype(np.int64))
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(pool, size=min(DUMP_SAMPLE, pool), replace=False))
    budget = (DUMP_MAX_BYTES - 16 * pool) // 4             # float32 per archive byte; the two index arrays are float64
    keep, total = [], 0
    for i in pick:
        if total + int(sizes[i]) > budget:
            continue
        keep.append(int(i))
        total += int(sizes[i])
    parts = [d_out[int(ooff[i]):int(ooff[i + 1])].cpu().numpy() for i in keep]
    sample = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "archive_block_sizes.npy"), sizes.astype(np.float64))
    np.save(os.path.join(out_dir, "archive_sample_blocks.npy"), np.asarray(keep, dtype=np.float64))
    np.save(os.path.join(out_dir, "archive_sample_bytes.npy"), sample.astype(np.float32))


def measure_config(rig: Rig, cfg_id: str, steps: int, warmup: int, batch_blocks: int = 0, sample_clocks: bool = False,
                   timed_decompress_reps: int = 1, warm_host_path: bool = True, dump_dir: str | None = None):
    """One config on this rank's GPU: device-resident compress (CUDA events), e2e compress and e2e decompress through the
    host-buffer ABI (pinned buffers, copies inside the timed region), round trip checked.  With `dump_dir`, rank 0 writes
    what the last timed device-resident step returned (dump_outputs)."""
    import torch
    from tools import synth
    z, ctx, dev, world = rig.z, rig.ctx, rig.dev, rig.world
    cfg = CONFIGS[cfg_id]
    bs = cfg["block"]
    how, arg = cfg["how"]
    hdr, pcomp, margs = model_of(cfg)
    state = z.device_state_bytes(hdr, False, bs)
    free, _ = torch.cuda.mem_get_info()
    if batch_blocks:
        B = batch_blocks
    else:
        io_per_block = bs * 6                         # input + slots + out + pre-processing work, device resident path
        B = int((free - (3 << 30)) // (state + io_per_block))
        B = max(1, min(B, cfg["max_blocks"]))
        try:                                          # one wave of the role-split encoder, when it applies
            ep = z.encoder_plan(hdr)
            if ep["applies"]:
                B = min(B, ep["blocks_per_sm"] * torch.cuda.get_device_properties(rig.local).multi_processor_count)
        except Exception:
            pass
    first = (rig.rank * B) % TOTAL_BLOCKS             # weak scaling: every GPU codes a full wave of its own blocks

    host_in = torch.empty(B * bs, dtype=torch.uint8).pin_memory()
    synth.fill(host_in.numpy(), cfg["kind"], first, B, bs)
    offs = np.arange(0, (B + 1) * bs, bs, dtype=np.uint64)
    out_cap = B * (bs + bs // 4 + 8192) + len(pcomp) * B
    host_out = torch.empty(out_cap, dtype=torch.uint8).pin_memory()
    d_in = host_in.to(dev, non_blocking=False)
    d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
    in_bytes = B * bs

    def step_device():
        return ctx.compress_blocks_model_dev(d_in.data_ptr(), offs, hdr, d_out.data_ptr(), out_cap, pcomp=pcomp, args=margs)

    def step_host():
        if how == "level":
            return ctx.compress_blocks_level(host_in.numpy(), offs, arg, out=host_out.numpy())
        return ctx.compress_blocks(host_in.numpy(), offs, arg, out=host_out.numpy())

    for _ in range(warmup):
        ooff = step_device()
    st = ctx.stats()
    resident = st.resident_blocks

    # ---- timed: device-resident path ----
    sampler = ClockSampler(rig.local) if sample_clocks else None
    rig.barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    codec_ms, kern_ms = [], []
    launches = 0
    e0.record(rig.stream)
    for _ in range(steps):
        ooff = step_device()
        s = ctx.stats()
        codec_ms.append(s.codec_kernel_ms)
        kern_ms.append(s.kernel_ms)
        launches += s.launches
    e1.record(rig.stream)
    rig.barrier()
    clocks = sampler.stop() if sampler else None
    t_dev = rig.max_time(e0.elapsed_time(e1) / 1e3)
    value = world * steps * in_bytes / 1e6 / t_dev
    ratio = float(ooff[B]) / in_bytes
    if dump_dir and rig.rank == 0:
        dump_outputs(dump_dir, d_out, ooff, B)
    del d_out
    del d_in
    torch.cuda.empty_cache()

    # ---- timed: end to end through the host-buffer ABI ----
    if warm_host_path:
        archive, hoff = step_host()        # warm the host path (pinned buffers, staging)
    rig.barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(steps):
        archive, hoff = step_host()
        s = ctx.stats()
        h2d += s.h2d_bytes
        d2h += s.d2h_bytes
        launches += s.launches
    torch.cuda.synchronize()
    t_e2e = rig.max_time(time.perf_counter() - t0)
    e2e_value = world * steps * in_bytes / 1e6 / t_e2e

    # ---- decompression of the same batch: e2e (host archive in, restored bytes out, pinned) ----
    back = torch.empty(in_bytes + 64, dtype=torch.uint8).pin_memory()
    out, o2, sha, bst = ctx.decompress_blocks(archive, hoff, out=back.numpy())        # warm-up + check of the whole batch
    ok = bool(np.array_equal(out, host_in.numpy())) and set(sha.tolist()) == {1}
    # one step of the decode direction = one resident wave of the DECODER (it holds fewer blocks per SM than the encoder for
    # some models; a batch of 1.09 waves would time a second, nearly empty wave at the first one's full latency)
    Bd = min(B, int(ctx.stats().resident_blocks) or B)
    dec_bytes = Bd * bs
    d_arc, d_off = archive[:int(hoff[Bd])], hoff[:Bd + 1]
    rig.barrier()
    t0 = time.perf_counter()
    dk_ms, dp_ms, dall_ms = [], [], []
    for _ in range(max(1, timed_decompress_reps)):
        out, o2, sha, bst = ctx.decompress_blocks(d_arc, d_off, out=back.numpy())
        s = ctx.stats()
        launches += s.launches
        dk_ms.append(s.codec_kernel_ms); dp_ms.append(s.post_kernel_ms); dall_ms.append(s.kernel_ms)
    torch.cuda.synchronize()
    t_d = rig.max_time(time.perf_counter() - t0) / max(1, timed_decompress_reps)
    ok = ok and bool(np.array_equal(out, host_in.numpy()[:dec_bytes])) and set(sha.tolist()) == {1}
    sd = ctx.stats()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    A = algorithmic_bytes(hdr, state, bs, ratio, margs[1] & 3)
    k_ms = sum(codec_ms) / len(codec_ms) if hdr[6] else sum(kern_ms) / len(kern_ms)
    dk = sum(dk_ms) / len(dk_ms) if hdr[6] else sum(dall_ms) / len(dall_ms)
    dec = {"e2e_value": world * dec_bytes / 1e6 / t_d, "unit": "MB/s", "blocks_per_gpu": Bd, "codec_kernel_ms": sum(dk_ms) / len(dk_ms),
           "post_kernel_ms": sum(dp_ms) / len(dp_ms), "kernel_ms": sum(dall_ms) / len(dall_ms),
           "kernel": sd.kernel.decode(errors="replace"), "resident_blocks": int(sd.resident_blocks),
           "post_native_blocks": int(sd.post_native_blocks), "post_interpreted_blocks": int(sd.post_interpreted_blocks),
           "round_trip_identical": ok, "sha1_verified_blocks": int((sha == 1).sum()), "in_bytes": dec_bytes,
           "roofline": {"bound": "hbm", "achieved": A * dec_bytes / (dk / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": A * dec_bytes / (dk / 1e3) / 1e9 / peak, "traffic": None, "algorithmic_bytes_per_input_byte": A,
                        "kernel_ms": dk}}
    res = {"config_id": cfg_id, "B": B, "block_bytes": bs, "in_bytes": in_bytes, "value": value, "t_dev": t_dev,
           "e2e_value": e2e_value, "h2d": h2d // max(steps, 1), "d2h": d2h // max(steps, 1), "launches": launches, "clocks": clocks,
           "ratio": ratio, "resident": int(resident), "state": int(st.state_bytes_per_block), "kernel": st.kernel.decode(errors="replace"),
           "kernel_ms": k_ms, "all_kernels_ms": sum(kern_ms) / len(kern_ms), "A": A, "peak": peak, "peak_measured": "hbm_gbs" in peaks,
           "decompress": dec, "archive": archive, "hoff": hoff, "host_in": host_in}
    return res


def summarise(r, world):
    """The per-config entry of the `configs` key."""
    ach = r["A"] * r["in_bytes"] / (r["kernel_ms"] / 1e3) / 1e9
    return {"workload": CONFIGS[r["config_id"]]["what"], "blocks_per_gpu": r["B"], "block_bytes": r["block_bytes"],
            "compress": {"value": r["value"], "e2e_value": r["e2e_value"], "unit": "MB/s", "kernel": r["kernel"], "kernel_ms": r["kernel_ms"],
                         "all_kernels_ms": r["all_kernels_ms"], "resident_blocks": r["resident"]},
            "decompress": {k: v for k, v in r["decompress"].items() if k != "roofline"},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": r["peak"], "unit": "GB/s", "frac": ach / r["peak"], "traffic": None,
                         "algorithmic_bytes_per_input_byte": r["A"]},
            "decompress_roofline": r["decompress"]["roofline"],
            "compression_ratio": r["ratio"], "state_bytes_per_block": r["state"], "n_gpus": world}


def c5_sweep(rig: Rig, full: bool = False):
    """BASELINE configs[4] / SURVEY 8d C5: mixed-method archives (equal quarters of mid.cfg, bit-packed LZ77 stored, byte LZ77 + CM
    chain, BWT blocks, interleaved) at four block payloads, decompressed through the host-buffer ABI.  The archives are written by
    this library (byte-identical to the oracle's, tests/test_gpu_parity.py)."""
    import torch
    from tools import synth
    z, ctx = rig.z, rig.ctx
    rows = []
    # about 1 GB of blocks per payload size; a block is restored at the speed of its own serial bit chain whatever the batch, so
    # the 16 MB leg takes minutes (a 16 MB mid.cfg block: ~40 s to code, ~90 s to decode) and runs only with --config C5
    legs = ((262144, 1024), (BLOCK, 256), (BLOCK_4MB, 64)) + (((BLOCK_16MB, 16),) if full else ())
    for bs, per_method in legs:
        a0 = 0 if bs <= BLOCK else (2 if bs == BLOCK_4MB else 4)
        groups = [("level", 2, "mixed"), ("method", lz_method(a0), "mixed"), ("method", lzcm_method(a0), "mixed"), ("method", bwt_method(a0), "text")]
        arcs, datas = [], []
        for gi, (how, arg, kind) in enumerate(groups):
            data = synth.blocks(kind, (rig.rank * 4 + gi) * per_method % TOTAL_BLOCKS, per_method, bs)
            offs = np.arange(0, (per_method + 1) * bs, bs, dtype=np.uint64)
            arc, ooff = (ctx.compress_blocks_level(data, offs, arg) if how == "level" else ctx.compress_blocks(data, offs, arg))
            arcs.append((arc.copy(), ooff)); datas.append(data)
        # interleave: block i of every method in turn
        pieces, plain = [], []
        for i in range(per_method):
            for gi in range(4):
                arc, ooff = arcs[gi]
                pieces.append(arc[int(ooff[i]):int(ooff[i + 1])])
                plain.append(datas[gi][i * bs:(i + 1) * bs])
        total_arc = sum(p.size for p in pieces)
        h_arc = torch.empty(total_arc, dtype=torch.uint8).pin_memory()
        np.concatenate(pieces, out=h_arc.numpy())
        aoff = np.concatenate([[0], np.cumsum([p.size for p in pieces])]).astype(np.uint64)
        n_out = 4 * per_method * bs
        back = torch.empty(n_out + 64, dtype=torch.uint8).pin_memory()
        out, o2, sha, bst = ctx.decompress_blocks(h_arc.numpy(), aoff, out=back.numpy())         # warm-up (NVRTC, buffers) + check
        ok = bool(np.array_equal(out, np.concatenate(plain))) and set(sha.tolist()) == {1}
        rig.torch.cuda.synchronize()
        t0 = time.perf_counter()
        out, o2, sha, bst = ctx.decompress_blocks(h_arc.numpy(), aoff, out=back.numpy())
        rig.torch.cuda.synchronize()
        t = time.perf_counter() - t0              # this rank's time; main() takes the maximum over the ranks (one collective, outside)
        st = ctx.stats()
        rows.append({"block_bytes": bs, "blocks_per_gpu": 4 * per_method, "methods": ["mid.cfg", lz_method(a0), lzcm_method(a0), bwt_method(a0)],
                     "seconds": t, "out_bytes_per_gpu": n_out,
                     "decompress_e2e_value": rig.world * n_out / 1e6 / t, "unit": "MB/s", "archive_bytes_per_gpu": int(total_arc),
                     "round_trip_identical": ok, "n_gpus": rig.world,
                     "post_native_blocks_last_group": int(st.post_native_blocks)})
        del h_arc, back
    return rows


def reduce_max_list(times, rig):
    tt = rig.torch.tensor(times, dtype=rig.torch.float64, device=rig.dev)
    rig.dist.all_reduce(tt, op=rig.dist.ReduceOp.MAX)
    return [float(x) for x in tt.tolist()]


def finish_c5(sweep, err, world, nlegs, full, reduce_max):
    """One collective for the whole sweep, entered by every rank whatever happened to it (a rank that failed contributes an
    infinite time): the slowest rank's time per leg decides the whole-job MB/s."""
    times = reduce_max([sweep[k]["seconds"] if k < len(sweep) else 1e30 for k in range(nlegs)])
    if err is not None or max(times) >= 1e29:
        return {"error": err or "a rank failed"}
    for k, row in enumerate(sweep):
        row["seconds"] = times[k]
        row["decompress_e2e_value"] = world * row["out_bytes_per_gpu"] / 1e6 / times[k]
    return {"workload": "configs[4]: mixed-method archive decompression sweep (mid.cfg / LZ77 stored / LZ77+CM / BWT blocks interleaved)",
            "sweep": sweep,
            "note": None if full else "the 16,773,120-byte leg runs with --config C5 (profiles/ holds the last full sweep)"}


def library_multi_gpu(rig: Rig, cfg_id: str, B: int):
    """The north-star's host call: ONE context on all N GPUs of the box, one zpq_compress_blocks_level / zpq_decompress_blocks
    call with host buffers; the library partitions the blocks over the devices and reassembles archives / restored bytes in block
    order (replaces the loops of LibZPAQ.cs:100-107 and :65-79).  Rank 0 drives it while the other ranks wait on the host."""
    import torch
    from tools import synth
    z = rig.z
    world = rig.world
    res = None
    rig.close()                              # every rank gives its GPU back
    if rig.host_group is not None:
        rig.dist.barrier(group=rig.host_group)
    if rig.rank == 0:
        cfg = CONFIGS[cfg_id]
        bs = cfg["block"]
        how, arg = cfg["how"]
        try:                                 # the leg pins input + archive + restored bytes of ALL devices on this one host
            import psutil
            room = int(0.45 * psutil.virtual_memory().available // (3.4 * bs * world))
            B = max(1, min(B, room))
        except Exception:
            pass
        nb = B * world
        wave = torch.empty(B * bs, dtype=torch.uint8)
        synth.fill(wave.numpy(), cfg["kind"], 0, B, bs)
        host_in = torch.empty(nb * bs, dtype=torch.uint8).pin_memory()
        for k in range(world):
            host_in[k * B * bs:(k + 1) * B * bs] = wave          # the wave of device 0 repeated for every device (same bytes per GPU)
        offs = np.arange(0, (nb + 1) * bs, bs, dtype=np.uint64)
        host_out = torch.empty(nb * (bs + bs // 4 + 8192), dtype=torch.uint8).pin_memory()
        back = torch.empty(nb * bs + 64, dtype=torch.uint8).pin_memory()
        with z.Context(list(range(world))) as ctx:
            run = (lambda: ctx.compress_blocks_level(host_in.numpy(), offs, arg, out=host_out.numpy())) if how == "level" else \
                  (lambda: ctx.compress_blocks(host_in.numpy(), offs, arg, out=host_out.numpy()))
            arc, ooff = run()
            t0 = time.perf_counter(); arc, ooff = run(); tc = time.perf_counter() - t0
            # ordered reassembly: the blocks of every device's wave are the same bytes, so every wave's archive must equal the first
            per = int(ooff[B])
            ordered = all(int(ooff[(k + 1) * B]) - int(ooff[k * B]) == per and
                          np.array_equal(arc[int(ooff[k * B]):int(ooff[(k + 1) * B])], arc[:per]) for k in range(world))
            out, o2, sha, bst = ctx.decompress_blocks(arc, ooff, out=back.numpy())
            t0 = time.perf_counter(); out, o2, sha, bst = ctx.decompress_blocks(arc, ooff, out=back.numpy()); td = time.perf_counter() - t0
            ok = bool(np.array_equal(out, host_in.numpy())) and set(sha.tolist()) == {1}
        res = {"devices": world, "blocks": nb, "blocks_per_device": B, "compress": {"e2e_value": nb * bs / 1e6 / tc, "unit": "MB/s", "archives_in_block_order": bool(ordered)},
               "decompress": {"e2e_value": nb * bs / 1e6 / td, "unit": "MB/s", "round_trip_identical": ok},
               "how": "one zpq_ctx over all devices, one call, host buffers (pinned), wall clock; rank 0 of %d" % world}
        del host_in, host_out, back
    if rig.host_group is not None:
        rig.dist.barrier(group=rig.host_group)
    rig.open()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2a", choices=sorted(CONFIGS) + ["C5"], help="which BASELINE config is the headline of the line (default C2a = configs[1])")
    ap.add_argument("--batch-blocks", type=int, default=0, help="blocks per GPU per step (0 = one resident wave)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the summary of the other configs (C1, C2b, C2c, C3, C4, C5)")
    ap.add_argument("--no-library-multi-gpu", action="store_true")
    ap.add_argument("--all-configs", action="store_true", help="N > 1: also run the C1 .. C4 summary on every rank")
    ap.add_argument("--configs", default="C1,C2a,C2b,C2c,C3,C4,C5", help="which configs the summary holds (comma separated)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step computed to DIR/*.npy (a fixed, seeded sample of the archive)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
        return

    rig = Rig()
    world, rank = rig.world, rig.rank
    head_id = args.config if args.config in CONFIGS else "C2a"
    r = measure_config(rig, head_id, args.steps, args.warmup, args.batch_blocks, sample_clocks=True, dump_dir=args.dump_outputs)
    k_ms = r["kernel_ms"]
    achieved = r["A"] * r["in_bytes"] / (k_ms / 1e3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if head_id == "C2a" and tj.get("dram_bytes_per_input_byte") is not None:
            traffic = tj["dram_bytes_per_input_byte"] * r["in_bytes"]
            if tj.get("decode_dram_bytes_per_input_byte") is not None:
                r["decompress"]["roofline"]["traffic"] = tj["decode_dram_bytes_per_input_byte"] * r["in_bytes"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": r["peak"], "unit": "GB/s", "frac": achieved / r["peak"],
                "traffic": traffic, "kernel": r["kernel"], "kernel_ms": k_ms,
                "algorithmic_bytes_per_input_byte": r["A"],
                "peak_source": "MEASURED_PEAKS.json (measured)" if r["peak_measured"] else "fallback 6650 GB/s",
                "traffic_source": "profiles/traffic.json: DRAM bytes per input byte from an ncu --set full capture of the same kernel, scaled to this launch" if traffic is not None else None,
                "note": "latency-bound: a dependent chain per role warp and block; the resident blocks are all that HBM and shared memory hold; see DESIGN.md 2.3"}
    B = r["B"]
    line = {
        "metric": CONFIGS[head_id]["metric"], "value": r["value"], "unit": "MB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["t_dev"] / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": workload_config(head_id, B, world),
        "e2e": {"value": r["e2e_value"], "unit": "MB/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
        "gpu_launches": r["launches"], "clocks": r["clocks"], "roofline": roofline,
        "compression_ratio": r["ratio"], "resident_blocks_per_gpu": r["resident"],
        "state_bytes_per_block": r["state"], "decompress": r["decompress"],
    }
    del r

    configs = {}
    if not args.no_configs:
        for cid in ("C1", "C2a", "C2b", "C2c", "C3", "C4"):
            if cid == head_id or args.config == "C5" or cid not in args.configs.split(","):   # --config C5: the headline line plus the FULL sweep, nothing else
                continue
            if world > 1 and not args.all_configs:          # under torchrun: headline + C5 sweep + library leg (the per-config
                continue                                    # summary is a one-GPU table; --all-configs runs it on every rank)
            try:
                rig.close(); rig.open()                 # the library's buffers are grow-only: every config starts from an empty device
                rc = measure_config(rig, cid, 1, 1, warm_host_path=False)
                line["gpu_launches"] += rc["launches"]
                configs[cid] = summarise(rc, world)
                del rc
            except Exception as e:                      # a config that fails is reported, it does not take the headline down
                configs[cid] = {"error": str(e)[:300]}
        if "C5" in args.configs.split(",") or args.config == "C5":
            c5_full = args.config == "C5"
            nlegs = 4 if c5_full else 3
            try:
                rig.close(); rig.open()
                sweep = c5_sweep(rig, full=c5_full)
                c5_err = None
            except Exception as e:
                sweep, c5_err = [], str(e)[:300]
            configs["C5"] = finish_c5(sweep, c5_err, world, nlegs, c5_full,
                                      (lambda t: reduce_max_list(t, rig)) if world > 1 else (lambda t: t))
    lib_multi = None
    if world > 1 and not args.no_library_multi_gpu:
        try:
            lib_multi = library_multi_gpu(rig, head_id, B)
        except Exception as e:
            lib_multi = {"error": str(e)[:300]}

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            base = cpu_baseline(head_id)
            line["cpu_baseline"] = base
            if base.get("decompress_value"):
                line["decompress"]["vs_cpu"] = line["decompress"]["e2e_value"] / base["decompress_value"]
                line["decompress"]["cpu_value"] = base["decompress_value"]
                line["decompress"]["cpu_kind"] = base.get("decompress_kind")
            for cid, c in configs.items():
                if cid in CONFIGS and "error" not in c:
                    try:
                        c["cpu_baseline"] = cpu_baseline(cid, seconds_budget=12.0, max_threads=16 if CONFIGS[cid]["block"] > BLOCK else None)
                    except Exception as e:
                        c["cpu_baseline"] = {"error": str(e)[:200]}
        if configs:
            line["configs"] = configs
        if lib_multi is not None:
            line["library_multi_gpu"] = lib_multi
        _emit(line)
    if world > 1:
        rig.dist.barrier()
        rig.dist.destroy_process_group()


def _emit(obj):
    """Write the one JSON line to the REAL stdout (libraries such as NCCL print banners to fd 1: it is parked on
    stderr for the whole run, see the bottom of this file)."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


if __name__ == "__main__":
    # stdout carries exactly one JSON line: everything else that is written to fd 1 (e.g. "NCCL version ...") goes to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    main()
