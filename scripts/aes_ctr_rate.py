"""AES-CTR rate of the library on one GPU (libzpaq AES_CTR::encrypt, zpq_aes_ctr_dev / zpq_aes_ctr).

    python scripts/aes_ctr_rate.py [--gib 4] [--reps 5] [--out FILE]

Device-resident: zpq_aes_ctr_dev over a buffer larger than L2 (default 4 GiB) for 128- and 256-bit keys, warmed up, timed
with CUDA events around `reps` calls on a torch stream the context is set to run on, plus the kernel time the library
reports.  Host-buffer: zpq_aes_ctr over the same size from pinned and from pageable memory (wall clock around the call,
which returns when the bytes are back).  The HBM share counts 2 bytes of traffic per byte (read + write) against the
6553.3 GB/s measured on a B200.  Prints the card's name, power limit and maximum SM clock from the same run.  Fails
when there is no GPU."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBPS = 6553.3   # measured copy bandwidth of one B200


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("aes_ctr_rate: no CUDA device (the measurement has no CPU form)")
    from zpaqsharp_b200 import libzpaq as z

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    say("card: " + (card[1] if len(card) > 1 else "?") + "   (" + (card[0] if card else "") + ")")
    n = int(a.gib * (1 << 30))
    say("buffer: %d bytes (%.2f GiB), larger than the 126 MB L2; %d timed calls per line after 2 warm-up calls" % (n, n / (1 << 30), a.reps))

    with z.Context([0]) as ctx:
        d = torch.zeros(n, dtype=torch.uint8, device="cuda")
        stream = torch.cuda.Stream()                  # a stream of its own: the events and the library's kernels share it
        torch.cuda.synchronize()
        ctx.set_stream(stream.cuda_stream)
        say("\ndevice-resident (zpq_aes_ctr_dev)")
        say("%-8s %10s %10s %12s %10s" % ("key", "GB/s", "kernel GB/s", "kernel ms", "HBM share"))
        for keylen in (16, 32):
            key, iv = bytes(range(keylen)), bytes(range(8))
            for _ in range(2):
                ctx.aes_ctr_dev(d.data_ptr(), n, key, iv, 0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            kms = []
            e0.record(stream)
            for r in range(a.reps):
                ctx.aes_ctr_dev(d.data_ptr(), n, key, iv, 16 * r)
                kms.append(ctx.stats().kernel_ms)
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / a.reps
            kms_min = min(kms)
            gbps = n / ms / 1e6
            say("AES-%-4d %10.1f %10.1f %12.3f %9.1f%%" % (8 * keylen, gbps, n / kms_min / 1e6, kms_min, 100 * 2 * gbps / HBM_GBPS))
            assert ctx.stats().kernel.decode() == "aes_ctr/%d" % (8 * keylen)
        ctx.set_stream(None)
        del d
        torch.cuda.empty_cache()

        say("\nhost buffer (zpq_aes_ctr: copy in, kernel, copy back in 1 GiB chunks, one stream)")
        say("%-8s %-9s %10s %10s %10s %10s" % ("key", "memory", "GB/s", "h2d ms", "kernel ms", "d2h ms"))
        pinned = torch.zeros(n, dtype=torch.uint8).pin_memory().numpy()
        pageable = np.zeros(n, dtype=np.uint8)
        for keylen in (16, 32):
            key, iv = bytes(range(keylen)), bytes(range(8))
            for name, buf in (("pinned", pinned), ("pageable", pageable)):
                ctx.aes_ctr(buf, key, iv, 0)
                best = None
                for _ in range(max(2, a.reps // 2)):
                    t = time.perf_counter()
                    ctx.aes_ctr(buf, key, iv, 0)
                    dt = time.perf_counter() - t
                    if best is None or dt < best[0]:
                        s = ctx.stats()
                        best = (dt, s.h2d_ms, s.kernel_ms, s.d2h_ms)
                say("AES-%-4d %-9s %10.1f %10.1f %10.1f %10.1f" % (8 * keylen, name, n / best[0] / 1e9, best[1], best[2], best[3]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
