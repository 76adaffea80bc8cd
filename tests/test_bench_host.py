"""Host-side pieces of bench.py that run without a GPU: the CPU baseline's reference codec (the reference's Compressor /
Decompresser text from oracle/_ref) must agree with the oracle and round-trip, and the reference arm must print the one
JSON line the bench contract asks for."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_codec_of_the_cpu_baseline_matches_oracle_and_round_trips():
    import bench
    from oracle import pyoracle as po
    from tools import synth
    codec = bench._reference_block_codec()
    if codec is None:
        pytest.skip("oracle/_ref fragments not available")
    comp, decomp = codec
    for n in (0, 1, 40000):
        data = synth.blocks("mixed", 5, 1, max(n, 1)).tobytes()[:n]
        arc = comp(data)
        assert arc == po.compress_block_level(data, bench.LEVEL)
        assert decomp(arc, len(data)) == data


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "MB/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_names_the_same_config_as_the_gpu_arm():
    """`same_config` of the driver compares the two arms' `config`: every key must be filled in on the CPU arm too."""
    import bench
    for cid in ("C2a", "C1", "C4"):
        cfg = bench.workload_config(cid, None, 1)
        assert cfg["batch_blocks_per_gpu"] and cfg["block_bytes"] == bench.CONFIGS[cid]["block"] and cfg["config_id"] == cid
        assert all(v is not None for v in cfg.values())
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--config", "C1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.strip()][0])
    assert d["impl"] == "reference" and d["config"]["config_id"] == "C1" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"


def test_algorithmic_bytes_of_the_survey():
    """SURVEY.md 8d: A(C2a) = 950 B per input byte, A(C1) = 66."""
    import bench
    from zpaqsharp_b200 import libzpaq as z
    hdr = z.builtin_model(2)
    a = bench.algorithmic_bytes(hdr, 111424512, bench.BLOCK, 0.3, 0)
    assert abs(a - 950) < 1.0
    text, args = z.make_config("x0,0c256,0,255,255")
    h1, _ = z.compile_config(text, args)
    assert abs(bench.algorithmic_bytes(h1, 1 << 20, bench.BLOCK, 0.3, 0) - 66.3) < 0.5


def test_dump_outputs_writes_a_fixed_sample_of_the_archive(tmp_path):
    """--dump-outputs: float arrays only, within 64 MB, the same sample whatever the batch size beyond the pool."""
    import numpy as np
    import torch
    import bench
    rng = np.random.default_rng(7)
    sizes = rng.integers(1, 5000, 400)
    ooff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    arc = torch.from_numpy(rng.integers(0, 256, int(ooff[-1]), dtype=np.uint8))
    bench.dump_outputs(str(tmp_path / "a"), arc, ooff, 400)
    bench.dump_outputs(str(tmp_path / "b"), arc, ooff, 300)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["archive_block_sizes.npy", "archive_sample_blocks.npy", "archive_sample_bytes.npy"]
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y)
    got = np.load(tmp_path / "a" / "archive_sample_bytes.npy")
    pick = np.load(tmp_path / "a" / "archive_sample_blocks.npy").astype(int)
    assert len(pick) == bench.DUMP_SAMPLE
    want = np.concatenate([arc.numpy()[int(ooff[i]):int(ooff[i + 1])] for i in pick])
    assert np.array_equal(got, want.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "archive_block_sizes.npy"), sizes[:bench.DUMP_POOL])
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= bench.DUMP_MAX_BYTES


def test_bench_rejects_zero_steps_and_dump_on_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert p.returncode == 2 and not p.stdout.strip(), p.stderr[-2000:]


def test_c5_sweep_is_reduced_with_one_collective_and_survives_a_failed_rank():
    import bench
    rows = [{"seconds": 2.0, "out_bytes_per_gpu": 10 ** 9, "decompress_e2e_value": 0.0}, {"seconds": 4.0, "out_bytes_per_gpu": 10 ** 9, "decompress_e2e_value": 0.0}]
    slower = lambda t: [max(x, 5.0) for x in t]                   # another rank needed 5 s for every leg
    out = bench.finish_c5([dict(r) for r in rows], None, 8, 2, False, slower)
    assert [round(r["decompress_e2e_value"]) for r in out["sweep"]] == [1600, 1600] and out["note"]
    out = bench.finish_c5([dict(r) for r in rows], None, 1, 2, True, lambda t: t)
    assert [round(r["decompress_e2e_value"]) for r in out["sweep"]] == [500, 250] and out["note"] is None
    assert "error" in bench.finish_c5(rows[:1], "out of memory", 2, 2, False, lambda t: t)
    assert "error" in bench.finish_c5([dict(r) for r in rows], None, 2, 2, False, lambda t: [1e30, 1e30])   # the other rank failed
