"""bench.py's contract on the CPU side: the reference arm prints one JSON line with the keys the driver reads, its
`ms_per_step` is the timed region that `value` is computed from, and the module's helpers that need no GPU behave.
One GPU test checks that --dump-outputs writes what the timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600,
                       cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-500:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--blocks", "512")
    assert d["impl"] == "reference" and d["unit"] == "MiB/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["dtype"] == "u8"
    assert d["config"]["blocks_per_gpu"] == 512 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["threads"] >= cb["cores"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "MiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # value and ms_per_step describe the same timed region: 512 blocks of 64 KiB = 32 MiB per step
    assert abs(d["value"] * d["ms_per_step"] / 1e3 - 32.0) < 0.01 * 32.0
    assert d["wall_ms_per_step"] >= d["ms_per_step"]


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1", "--blocks", "64"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_ncu_traffic_lookup_is_by_exact_kernel():
    sys.path.insert(0, ROOT)
    import bench
    got, src = bench.ncu_traffic("lz4_compress_blocks_gtab<unsigned short, 7, 1, 0>")
    assert src == "r2_ncu_summary.json" and 3.0e10 < got < 6.0e10           # dram read + write of the committed capture
    got2, src2 = bench.ncu_traffic("lz4_decompress_blocks<8, 0, 0, 1>")
    assert src2 == "r2_ncu_summary.json" and 2.0e9 < got2 < 5.0e9
    assert bench.ncu_traffic("lz4_compress_blocks_gtabg<8, 7, 1>") == (None, None)   # no capture of that kernel: no number


def test_workload_is_the_tiled_fixture():
    sys.path.insert(0, ROOT)
    import bench
    from lz4_flex_b200 import corpus
    w = bench.build_workload(8, 0)
    assert w.dtype == np.uint8 and w.size == 8 * 65536
    assert np.array_equal(w, corpus.tiled("compression_66k_JSON.txt", 8 * 65536))


def test_dump_outputs_files(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    idx = bench.dump_sample(bench.NBLOCKS_DEFAULT)
    assert np.array_equal(idx, bench.dump_sample(bench.NBLOCKS_DEFAULT)) and np.all(np.diff(idx) > 0)
    assert np.array_equal(bench.dump_sample(5), np.arange(5))
    nb, slot = 8, 16
    comp = np.arange(nb * slot, dtype=np.uint8).reshape(nb, slot)
    clen = np.arange(nb, dtype=np.int32) + 3
    back = np.full((nb, 4), 7, dtype=np.uint8)
    sel = np.array([1, 6])
    bench.dump_outputs(str(tmp_path), sel, comp[sel], clen, np.zeros(nb), back[sel], np.full(nb, 4), np.zeros(nb))
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert set(got) == {"sample_block_index", "compressed_len", "compress_status", "compressed_sample",
                        "decompressed_len", "decompress_status", "decompressed_sample"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["compressed_len"], clen)
    assert np.array_equal(got["compressed_sample"][0], np.where(np.arange(slot) < 4, comp[1], 0))
    assert np.array_equal(got["compressed_sample"][1], np.where(np.arange(slot) < 9, comp[6], 0))
    assert np.array_equal(got["decompressed_sample"], back[sel])
    # at the default batch the files stay under 64 MB in all
    k = bench.DUMP_SAMPLE_BLOCKS
    assert 4 * k * (72112 + 65536) + 8 * (4 * bench.NBLOCKS_DEFAULT + k) < 64 << 20


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_step(tmp_path):
    """bench.py --dump-outputs on a small batch: the files hold what the oracle computes for the same input."""
    sys.path.insert(0, ROOT)
    import bench
    import oracle
    nb = 256
    d = _run("--steps", "2", "--warmup", "1", "--blocks", str(nb), "--quick", "--no-frame", "--dump-outputs", str(tmp_path))
    assert d["quick"] is True
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    data = bench.build_workload(nb, 0).reshape(nb, bench.BLOCK)
    idx = bench.dump_sample(nb)
    assert np.array_equal(got["sample_block_index"], idx)
    assert not got["compress_status"].any() and not got["decompress_status"].any()
    assert np.array_equal(got["decompressed_len"], np.full(nb, bench.BLOCK))
    assert np.array_equal(got["decompressed_sample"], data[idx])
    want = [oracle.compress_block(data[i].tobytes()) for i in range(nb)]
    assert np.array_equal(got["compressed_len"], [len(w) for w in want])
    for row, i in zip(got["compressed_sample"], idx):
        w = np.frombuffer(want[i], dtype=np.uint8)
        assert np.array_equal(row[:w.size], w) and not row[w.size:].any()
