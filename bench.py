#!/usr/bin/env python
"""bench.py — LZ4 block compress+decompress throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference arm: CPU path on host cores
    python bench.py --steps K --dump-outputs DIR             # also write what the last timed step computed (DIR/*.npy)

Workload (BASELINE config 2): 16 384 independent 64 KiB blocks cut from compression_66k_JSON.txt tiled to
1 GiB, block format.  One STEP = compress all blocks, then decompress all of them (per rank).  N > 1 shards
blocks across ranks (every rank owns its own 16 384 blocks: weak scaling, no data-path collective; the
frame-mode gather of compressed chunks is measured separately with --workload frame).

value      = uncompressed MiB per second of the whole job (all ranks) over the compress+decompress step,
             inputs resident in HBM, timed with CUDA events, max over ranks.
e2e        = the same metric through the host-pointer C-ABI calls, H2D/D2H copies inside the timed region, measured two
             ways and both reported: one step at a time (compress call, then decompress call), and as a stream of batches
             (compress of batch k on one thread / context next to decompress of batch k-1 on another: the two calls use
             opposite directions of the PCIe link; K batches timed including fill and drain).  `e2e.value` is the better
             one and `e2e.mode` names it.
roofline   = dominant kernel (compress) against the measured HBM copy peak; the decompress kernel's roofline is
             reported beside it.
cpu_baseline = the C oracle (a restatement of lz4_flex's algorithm; Rust is not available) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 65536
NBLOCKS_DEFAULT = 16384
FIXTURE = "compression_66k_JSON.txt"
METRIC = "LZ4 block MiB/s (compress+decompress) at 1/2/4/8 B200 vs CPU; % HBM peak"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  NVML in-process at
    ~2 ms intervals (the timed region of the default run lasts ~0.25 s, too short for an `nvidia-smi -lms` loop to
    deliver samples); falls back to the nvidia-smi loop when pynvml is unavailable."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []
        self.nvml = None
        self.handle = None
        self.samples = []           # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(device).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.nvml, self.handle = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        n, h = self.nvml, self.handle
        while not self._stop.is_set():
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
                try:
                    why = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    why = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append((mhz, why))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.t.join(timeout=1)
            sm = [s[0] for s in self.samples]
            mask = 0
            for _, w in self.samples:
                mask |= w
            reasons = sorted(nm for bit, nm in self.BITS.items() if mask & bit)
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def ncu_traffic(kernel: str):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` — the name the launcher reported
    for this run (lz4b200_ctx_last_kernel) — from the committed ncu --set full summaries of this workload
    (profiles/r2_ncu_summary.json, then r1), or None when that exact kernel has no capture: a profile is never
    attributed to a kernel it was not taken from."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    norm = lambda n: n.replace("void ", "").split("(")[0].replace("lz4b200::", "").replace("(int)", "").replace("false", "0").replace("true", "1").replace(" ", "")
    for f in ("r2_ncu_summary.json", "r1_ncu_summary.json"):
        try:
            for e in json.load(open(os.path.join(ROOT, "profiles", f))):
                if norm(e.get("kernel", "")) == norm(kernel):
                    tot = 0.0
                    for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                        v, u = e[k].split()
                        tot += float(v) * unit[u]
                    return tot, f
        except Exception:                                       # noqa: BLE001
            pass
    return None, None


def build_workload(nblocks: int, rank: int):
    from lz4_flex_b200 import corpus
    total = nblocks * BLOCK
    src = np.frombuffer(corpus.load(FIXTURE), dtype=np.uint8)
    # rank r continues the tiling where rank r-1 stopped, so every rank has distinct block phases
    start = (rank * total) % src.size
    reps = -(-(total + start) // src.size)
    data = np.tile(src, reps)[start:start + total]
    return np.ascontiguousarray(data)


DUMP_SEED = 20260917
DUMP_SAMPLE_BLOCKS = 64                                 # 64 x (72112 + 65536) bytes as float32: 35 MB, under 64 MB in all


def dump_sample(nblocks: int) -> np.ndarray:
    """Indices of the blocks whose bytes --dump-outputs writes: a fixed, seeded sample, sorted."""
    rng = np.random.default_rng(DUMP_SEED)
    return np.sort(rng.choice(nblocks, size=min(nblocks, DUMP_SAMPLE_BLOCKS), replace=False))


def dump_outputs(path: str, idx, comp_rows, comp_len, comp_status, back_rows, back_len, back_status):
    """Writes what one compress+decompress step returned to its caller as float .npy files, so that two builds can be
    compared output for output: per-block lengths and statuses of every block, and the compressed and decompressed bytes
    of the sampled blocks `idx` (compressed rows zeroed past each block's length: those slot bytes are not output)."""
    os.makedirs(path, exist_ok=True)
    comp_rows = np.asarray(comp_rows, dtype=np.float32)
    comp_rows[np.arange(comp_rows.shape[1])[None, :] >= np.asarray(comp_len)[idx][:, None]] = 0
    arrays = {
        "sample_block_index": np.asarray(idx, dtype=np.float64),
        "compressed_len": np.asarray(comp_len, dtype=np.float64),
        "compress_status": np.asarray(comp_status, dtype=np.float64),
        "compressed_sample": comp_rows,
        "decompressed_len": np.asarray(back_len, dtype=np.float64),
        "decompress_status": np.asarray(back_status, dtype=np.float64),
        "decompressed_sample": np.asarray(back_rows, dtype=np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def host_topology():
    """(logical CPUs usable by this process, physical cores among them) — the reference arm reports both."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            pkg = open(f"/sys/devices/system/cpu/cpu{c}/topology/physical_package_id").read().strip()
            cid = open(f"/sys/devices/system/cpu/cpu{c}/topology/core_id").read().strip()
            cores.add((pkg, cid))
        except OSError:
            cores.add(("?", str(c)))
    return len(cpus), len(cores)


_POOLS = {}


def cpu_arm(data: np.ndarray, nblocks: int, threads: int, repeats: int):
    """The CPU implementation of the path (oracle/lz4_cpu_baseline.c: the restatement of lz4_flex's unsafe block path,
    byte-identical to the oracle) compress+decompress of `nblocks` blocks on a persistent pool of `threads` host
    threads; best of `repeats`."""
    import oracle
    if threads not in _POOLS:
        _POOLS[threads] = oracle.Pool(threads)
    pool = _POOLS[threads]
    slot = 72112
    offs = np.arange(nblocks, dtype=np.uint64) * BLOCK
    lens = np.full(nblocks, BLOCK, dtype=np.uint32)
    soff = np.arange(nblocks, dtype=np.uint64) * slot
    scap = np.full(nblocks, slot, dtype=np.uint32)
    key = ("bufs", nblocks, threads)
    if key not in _POOLS:
        # every buffer the workers stream through is first touched BY the workers (pool.copy), so its pages spread over the
        # host's NUMA nodes instead of all sitting on the node of this thread (measured: 9.5 vs 35 GiB/s decompress)
        comp = np.empty(nblocks * slot, dtype=np.uint8)
        back = np.empty(nblocks * BLOCK, dtype=np.uint8)
        src = np.empty(nblocks * BLOCK, dtype=np.uint8)
        pool.copy(comp); pool.copy(back); pool.copy(src, data[: nblocks * BLOCK])
        _POOLS[key] = (comp, back, src)
        pool.compress(src, offs, lens, comp, soff, scap)         # untimed warm-up pass
    comp, back, src = _POOLS[key]
    best = (1e30, 1e30)
    clen = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        clen, st = pool.compress(src, offs, lens, comp, soff, scap)
        t1 = time.perf_counter()
        olen, st2 = pool.decompress(comp, soff, clen, back, offs, lens)
        t2 = time.perf_counter()
        assert not st.any() and not st2.any()
        if (t2 - t0) < sum(best):
            best = (t1 - t0, t2 - t1)
    assert np.array_equal(back[: nblocks * BLOCK], data[: nblocks * BLOCK])
    mib = nblocks * BLOCK / 2**20
    return {"compress_mibs": mib / best[0], "decompress_mibs": mib / best[1], "roundtrip_mibs": mib / sum(best),
            "ratio": float(clen.astype(np.uint64).sum()) / (nblocks * BLOCK)}


def cpu_arm_fresh_process(nblocks: int):
    """The all-thread CPU baseline of the bench line, taken in a FRESH process (`bench.py --impl reference`): the same
    thing the driver's reference arm runs.  Measured in-process after the GPU phases (CUDA context, pinned buffers, an
    affinity binding undone) the same pool gave 10 GiB/s compress on a box where the fresh process gives 88 GiB/s."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
                            "--blocks", str(nblocks)], capture_output=True, text=True, timeout=600,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        d = json.loads(r.stdout.strip().splitlines()[-1])
        c = d["cpu_baseline"]
        return {"compress_mibs": c["compress_mibs"], "decompress_mibs": c["decompress_mibs"], "roundtrip_mibs": d["value"],
                "how": "fresh process (bench.py --impl reference --steps 3 --warmup 1), median of 3 steps"}
    except Exception:                                           # noqa: BLE001
        return None


def liblz4_anchor(data: np.ndarray, nblocks: int):
    """Sanity anchor (SURVEY.md §8d): system liblz4 (LZ4_compress_default / LZ4_decompress_safe), one thread, same
    blocks.  lz4_flex's README puts its unsafe path within ~10 % of C lz4.  Returns None when liblz4 is absent."""
    import ctypes
    try:
        L = ctypes.CDLL("liblz4.so.1")
    except OSError:
        return None
    L.LZ4_compress_default.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    L.LZ4_decompress_safe.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    L.LZ4_compressBound.argtypes = [ctypes.c_int]
    bound = L.LZ4_compressBound(BLOCK)
    comp = np.zeros(nblocks * bound, dtype=np.uint8)
    back = np.zeros(nblocks * BLOCK, dtype=np.uint8)
    clen = np.zeros(nblocks, dtype=np.int64)
    comp[::4096] = 1; back[::4096] = 1                       # pre-fault
    src, dst, bk = data.ctypes.data, comp.ctypes.data, back.ctypes.data
    best_c = best_d = 1e30
    for _ in range(2):
        t0 = time.perf_counter()
        for b in range(nblocks):
            clen[b] = L.LZ4_compress_default(src + b * BLOCK, dst + b * bound, BLOCK, bound)
        t1 = time.perf_counter()
        for b in range(nblocks):
            L.LZ4_decompress_safe(dst + b * bound, bk + b * BLOCK, int(clen[b]), BLOCK)
        t2 = time.perf_counter()
        best_c, best_d = min(best_c, t1 - t0), min(best_d, t2 - t1)
    if not np.array_equal(back, data[: nblocks * BLOCK]):
        return None
    mib = nblocks * BLOCK / 2**20
    return {"library": "liblz4 (system)", "threads": 1, "compress_mibs": mib / best_c, "decompress_mibs": mib / best_d,
            "ratio": float(clen.sum()) / (nblocks * BLOCK)}


def run_reference(args):
    """Reference arm: the CPU implementation of the path on all host threads (the C port of lz4_flex's unsafe path —
    no Rust toolchain exists here), same config as our arm: every step compresses and decompresses ALL blocks."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, cores = host_topology()
    nblocks = args.blocks
    data = build_workload(nblocks, 0)
    for _ in range(max(args.warmup, 1)):
        cpu_arm(data, nblocks, threads, 1)
    t0 = time.perf_counter()
    res = [cpu_arm(data, nblocks, threads, 1) for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    val = float(np.median([r["roundtrip_mibs"] for r in res]))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "MiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * (nblocks * BLOCK / 2**20) / val,
        "wall_ms_per_step": 1e3 * dt / max(args.steps, 1),     # includes the per-step verification of the round trip
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": f"{FIXTURE} tiled (deterministic corpus fixture, BASELINE config 2)",
        "config": {"workload": f"{args.blocks} x 64 KiB JSON blocks, block format, compress+decompress",
                   "block_bytes": BLOCK, "blocks_per_gpu": args.blocks},
        "cpu_baseline": {"value": val, "unit": "MiB/s", "cores": cores, "threads": threads, "kind": "port",
                         "sample": f"all {nblocks} blocks per step (same config as the GPU arm), compress+decompress, "
                                   f"{threads} persistent threads on {cores} physical cores, blocks handed out in chunks of 8",
                         "compress_mibs": float(np.median([r['compress_mibs'] for r in res])),
                         "decompress_mibs": float(np.median([r['decompress_mibs'] for r in res]))},
        "e2e": {"value": val, "unit": "MiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from lz4_flex_b200 import block

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # bind this rank (and the pinned staging buffers it allocates from here on) to its GPU's NUMA node
    from lz4_flex_b200 import numa
    ninfo = numa.bind_to_gpu_node(local)
    numa_rec = {k: v for k, v in ninfo.items() if k != "original_affinity"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    nb = args.blocks
    data = build_workload(nb, rank)
    ctx = block.Context(local)
    slot = 72112                                        # get_maximum_output_size(65536) = 72109, 16-byte aligned
    offs = np.arange(nb, dtype=np.uint64) * BLOCK
    lens = np.full(nb, BLOCK, dtype=np.uint32)
    soff = np.arange(nb, dtype=np.uint64) * slot
    scap = np.full(nb, slot, dtype=np.uint32)

    h_in = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
    h_in.numpy()[:] = data
    d_in = h_in.to(dev, non_blocking=True)
    d_comp = torch.zeros(nb * slot, dtype=torch.uint8, device=dev)
    d_back = torch.zeros(nb * BLOCK, dtype=torch.uint8, device=dev)
    enc = block.DeviceBatch(offs, lens, soff, scap, None, dev)
    dec = block.DeviceBatch(soff, lens, offs, lens, None, dev)
    dec.in_len = enc.out_len                             # decompress reads exactly what compress produced
    torch.cuda.synchronize()

    def step(events=None):
        if events is not None:
            events[0].record()
        enc.compress(d_in, d_comp, ctx)
        if events is not None:
            events[1].record()
        dec.decompress(d_comp, d_back, ctx)
        if events is not None:
            events[2].record()

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    # verification outside the timed region: statuses, exact round trip, oracle bytes on a sample
    assert int(enc.status.abs().sum()) == 0 and int(dec.status.abs().sum()) == 0, "block status != OK"
    assert torch.equal(d_back, d_in), "round trip differs from the input"
    clen = enc.out_len.cpu().numpy().astype(np.uint64)
    comp_bytes = int(clen.sum())
    if rank == 0:
        # every block of the batch against the oracle (all host threads), not a sample
        import oracle
        want = np.zeros(nb * slot, dtype=np.uint8)
        wlen, wst = oracle.compress_batch(data, offs, lens, want, soff, scap, os.cpu_count() or 1)
        assert np.array_equal(wlen.astype(np.uint64), clen), "compressed lengths differ from the oracle"
        got = d_comp.cpu().numpy().reshape(nb, slot)
        used = np.arange(slot, dtype=np.uint32)[None, :] < wlen[:, None]
        assert not ((got != want.reshape(nb, slot)) & used).any(), "compressed bytes differ from the oracle"
        del want, got, used

    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for k in range(args.steps):
        step(evs[k])
    t_end.record()
    torch.cuda.synchronize()
    k1_name, k2_name = _last_kernel(ctx, 0), _last_kernel(ctx, 1)       # what the launcher picked for the timed batches
    if args.dump_outputs and rank == 0:
        idx = dump_sample(nb)
        rows = torch.from_numpy(idx).to(dev)
        dump_outputs(args.dump_outputs, idx, d_comp.view(nb, slot)[rows].cpu().numpy(), enc.out_len.cpu().numpy(),
                     enc.status.cpu().numpy(), d_back.view(nb, BLOCK)[rows].cpu().numpy(), dec.out_len.cpu().numpy(),
                     dec.status.cpu().numpy())
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = t_start.elapsed_time(t_end)
    t_c = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
    t_d = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
    if world > 1:
        t = torch.tensor([elapsed_ms, t_c, t_d], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, t_c, t_d = [float(x) for x in t.cpu()]

    if args.quick:                                      # tuning aid: device-timed kernels only
        if rank == 0:
            print(json.dumps({"quick": True, "compress_ms": t_c, "decompress_ms": t_d,
                              "ms_per_step": elapsed_ms / args.steps}))
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- end-to-end through the host-pointer C ABI (pinned host buffers, copies inside the timed region) ----
    h_comp = torch.empty(comp_bytes + 4096, dtype=torch.uint8).pin_memory()
    h_back = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
    e2e_steps = max(1, min(args.steps, 5))
    e2e_t = []
    call_t = []
    for it in range(2 + e2e_steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out, ooff, olen = block.compress_batch(h_in.numpy(), offs, lens, None, out=h_comp.numpy(), ctx=ctx)
        t1 = time.perf_counter()
        block.decompress_batch(out, ooff, olen, h_back.numpy(), offs, lens, ctx=ctx)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if it >= 2:
            e2e_t.append(dt)
            call_t.append((t1 - t0, dt - (t1 - t0)))
    assert np.array_equal(h_back.numpy(), data)
    e2e_serial_s = float(np.mean(e2e_t))
    # what the PCIe link of THIS rank delivers while every rank copies at once (pinned, 1 GiB each way): the floor of the step
    link = {}
    for name, fn in (("h2d", lambda: d_in.copy_(h_in, non_blocking=True)), ("d2h", lambda: h_back.copy_(d_back, non_blocking=True))):
        ts = []
        for it in range(3):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        link[name + "_gbs"] = round(nb * BLOCK / min(ts[1:]) / 1e9, 2)
    # both directions at once (two streams): what a perfectly overlapped compress + decompress pipeline could count on
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
    ts = []
    for it in range(3):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(s_up):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_back.copy_(d_back, non_blocking=True)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    link["duplex_gbs_each_way"] = round(nb * BLOCK / min(ts[1:]) / 1e9, 2)

    # The same two C-ABI calls, used the way a streaming caller would: the batch is cut into chunks, one host
    # thread compresses chunk c+1 (context A) while another decompresses chunk c (context B), so the H2D-heavy
    # compress side and the D2H-heavy decompress side share the full-duplex PCIe link.  Every byte still makes the
    # whole trip host -> GPU compress -> host (compressed) -> GPU decompress -> host inside the timed region.
    import threading
    import queue as _queue
    ctx2 = block.Context(local, high_priority=True)      # decode kernels are short: let them jump the encoder's queue

    def pipelined(nchunks):
        per = -(-nb // nchunks)
        q = _queue.Queue()
        err = []

        def comp():
            try:
                pos = 0
                hc = h_comp.numpy()
                for b0 in range(0, nb, per):
                    b1 = min(nb, b0 + per)
                    o, ooff, olen = block.compress_batch(h_in.numpy(), offs[b0:b1], lens[b0:b1], None, out=hc[pos:], ctx=ctx)
                    used = int(ooff[-1]) + int(olen[-1])
                    q.put((b0, b1, pos, ooff, olen))
                    pos += used
            except Exception as e:                      # noqa: BLE001
                err.append(e)
            q.put(None)

        th = threading.Thread(target=comp)
        th.start()
        hc = h_comp.numpy()
        while True:
            it = q.get()
            if it is None:
                break
            b0, b1, pos, ooff, olen = it
            block.decompress_batch(hc[pos:], ooff, olen, h_back.numpy(), offs[b0:b1], lens[b0:b1], ctx=ctx2)
        th.join()
        if err:
            raise err[0]

    # A worker-pool caller (what a rayon-style user of the batch calls does): the batch is cut into chunks, `nc`
    # threads (one context each) take chunks in order and compress them, `nd` threads decompress each chunk as soon
    # as its compressed bytes are back on the host.  One call's tail (the last block's serial chain, ~5 ms, with the
    # H2D link idle) overlaps the next call's copies, and compress H2D runs next to decompress D2H on the duplex link.
    pool_ctx = {}
    h_comp_slots = None

    def pooled(nchunks, nc, nd):
        nonlocal h_comp_slots
        if h_comp_slots is None:
            h_comp_slots = torch.empty(nb * slot, dtype=torch.uint8).pin_memory()   # worst-case region per chunk
        per = -(-nb // nchunks)
        todo = _queue.Queue()
        done = _queue.Queue()
        for b0 in range(0, nb, per):
            todo.put((b0, min(nb, b0 + per)))
        err = []
        hs = h_comp_slots.numpy()

        def cw(i):
            c = pool_ctx.setdefault(("c", i), block.Context(local))
            try:
                while True:
                    try:
                        b0, b1 = todo.get_nowait()
                    except _queue.Empty:
                        break
                    o, ooff, olen = block.compress_batch(h_in.numpy(), offs[b0:b1], lens[b0:b1], None,
                                                         out=hs[b0 * slot:b1 * slot], ctx=c)
                    done.put((b0, b1, ooff, olen))
            except Exception as e:                      # noqa: BLE001
                err.append(e)

        def dw(i):
            c = pool_ctx.setdefault(("d", i), block.Context(local, high_priority=True))
            try:
                while True:
                    it = done.get()
                    if it is None:
                        break
                    b0, b1, ooff, olen = it
                    block.decompress_batch(hs[b0 * slot:b1 * slot], ooff, olen, h_back.numpy(), offs[b0:b1], lens[b0:b1], ctx=c)
            except Exception as e:                      # noqa: BLE001
                err.append(e)

        cws = [threading.Thread(target=cw, args=(i,)) for i in range(nc)]
        dws = [threading.Thread(target=dw, args=(i,)) for i in range(nd)]
        for t in cws + dws:
            t.start()
        for t in cws:
            t.join()
        for _ in dws:
            done.put(None)
        for t in dws:
            t.join()
        if err:
            raise err[0]

    best_chunks, e2e_s, e2e_how = 1, e2e_serial_s, "one call each, back to back"
    # measured on B200 (profiles/r2_e2e_callers.txt): serial 48.6 ms; pipelined x2/x4/x8 51.6 / 54.3 / 66.7; pooled (8,2,1) /
    # (8,3,2) / (16,3,2) / (16,4,2) 63.9 / 59.9 / 64.7 / 63.8 — the encoder's persistent CTAs leave the decoder no warp slots,
    # so overlapping the two calls only adds per-call tails.  Two probes stay so that the record shows the comparison was made.
    cands = [("pipelined", (2,)), ("pooled", (8, 3, 2))]
    if os.environ.get("LZ4B200_E2E_POOL"):               # tuning aid: "chunks,compress_threads,decompress_threads;..."
        cands = [("pooled", tuple(int(v) for v in c.split(","))) for c in os.environ["LZ4B200_E2E_POOL"].split(";")]
    for kind, cfg in (cands if nb >= 4096 else []):
        ts = []
        for it in range(2 + e2e_steps):
            h_back.numpy()[::4096] = 0
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            (pipelined if kind == "pipelined" else pooled)(*cfg)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it >= 2:
                ts.append(dt)
        assert np.array_equal(h_back.numpy(), data)
        if float(np.mean(ts)) < e2e_s:
            best_chunks, e2e_s = cfg[0], float(np.mean(ts))
            e2e_how = (f"{cfg[0]} chunks, one compress thread feeding one decompress thread" if kind == "pipelined" else
                       f"{cfg[0]} chunks, {cfg[1]} compress threads + {cfg[2]} decompress threads (one context each)")
        if rank == 0 and os.environ.get("LZ4B200_DEBUG"):
            print(f"# e2e {kind} {cfg}: {1e3 * float(np.mean(ts)):.2f} ms (serial {1e3 * e2e_serial_s:.2f} ms)", file=sys.stderr)
    pool_ctx.clear()
    h_comp_slots = None

    # ---- a STREAM of batches through the same two calls: while batch k is compressed (thread A, context 1: 1 GiB up, 0.25 GiB
    # down) batch k-1 is decompressed (thread B, context 2: 0.25 GiB up, 1 GiB down).  Every batch still makes the whole trip
    # host -> compress -> host -> decompress -> host; the two calls of one tick use opposite directions of the duplex link
    # and no call is cut into chunks (no extra tails).  Timed over K batches INCLUDING the fill and drain ticks (K + 1 ticks).
    h_comp2 = torch.empty(comp_bytes + 4096, dtype=torch.uint8).pin_memory()

    def stream(K):
        bufs = [h_comp.numpy(), h_comp2.numpy()]
        res = [None, None]
        err = []

        def comp(k):
            try:
                res[k & 1] = block.compress_batch(h_in.numpy(), offs, lens, None, out=bufs[k & 1], ctx=ctx)
            except Exception as e:                      # noqa: BLE001
                err.append(e)

        for k in range(K + 1):
            th = None
            if k < K:
                th = threading.Thread(target=comp, args=(k,))
                th.start()
            try:
                if k >= 1:
                    o, ooff, olen = res[(k - 1) & 1]
                    block.decompress_batch(o, ooff, olen, h_back.numpy(), offs, lens, ctx=ctx2)
            finally:
                if th is not None:
                    th.join()                               # never leave the compress thread running on `ctx`
            if err:
                raise err[0]

    stream_rec, stream_failed = None, None
    if nb >= 4096:
        K = 4 * e2e_steps                               # 20 batches by default: fill + drain add one tick to K
        # (free-running variants — no join per tick, one or two compress threads — were slower at N=1, 39.8-41.4 ms vs 37.6,
        # and the two-compress-thread one once handed the decoder an incomplete buffer at N=8: not kept.)
        ts, stream_err = [], None
        for it in range(3):                                 # a failure on one rank must not leave the others in a collective
            h_back.numpy()[::4096] = 0
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            try:
                stream(K)
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) / K)
                if not np.array_equal(h_back.numpy(), data):
                    stream_err = "round trip differs from the input"
            except Exception as e:                          # noqa: BLE001
                stream_err = f"{type(e).__name__}: {e}"
                ts.append(1e30)
        stream_s, stream_how = float(min(ts[1:])), "both calls joined per tick"
        stream_local = stream_s
        ok = 0.0 if stream_err else 1.0
        if world > 1:
            t = torch.tensor([stream_s, -ok], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            stream_s, ok = float(t.cpu()[0]), -float(t.cpu()[1])
        if ok < 1.0:                                        # reported, never counted
            stream_rec, stream_s = None, 1e30
            stream_failed = stream_err or "failed on another rank"
            print(f"# rank {rank}: e2e stream mode failed: {stream_failed}", file=sys.stderr)
        else:
            stream_failed = None
            stream_rec = {"value": world * (nb * BLOCK / 2**20) / stream_s, "unit": "MiB/s", "ms_per_batch": 1e3 * stream_s, "batches": K,
                          "how": f"compress(batch k) on its own host thread(s) / context(s) while earlier batches are decompressed on "
                                 f"another ({stream_how}); {K} batches timed including fill and drain; every batch makes the whole round trip"}
        if rank == 0 and stream_rec and os.environ.get("LZ4B200_DEBUG"):
            print(f"# e2e stream of {K} batches: {1e3 * stream_s:.2f} ms per batch (serial {1e3 * e2e_serial_s:.2f} ms)", file=sys.stderr)
    del h_comp2
    per_rank = None
    if world > 1:
        # every rank's own e2e time and NUMA placement go into the record (which ranks are the slow ones, and where they sit)
        mine = {"rank": rank, "e2e_ms": round(1e3 * e2e_s, 2), "stream_ms": round(1e3 * stream_local, 2) if stream_rec else None,
                "compress_call_ms": round(1e3 * float(np.mean([c for c, _ in call_t])), 2),
                "decompress_call_ms": round(1e3 * float(np.mean([d for _, d in call_t])), 2), **link, **numa_rec}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        t = torch.tensor([e2e_s, e2e_serial_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s, e2e_serial_s = float(t.cpu()[0]), float(t.cpu()[1])
    desc_bytes = nb * (8 + 4 + 8 + 4)
    h2d = nb * BLOCK + comp_bytes + 2 * desc_bytes
    d2h = comp_bytes + nb * BLOCK + nb * (4 + 4 + 8) + nb * (4 + 4 + 8)

    # ---- the multi-GPU path of the north star (BASELINE config 4), measured at every N as a second record ----------
    del d_comp, d_back, h_comp, h_back
    torch.cuda.empty_cache()
    frame_rec = None
    if not args.no_frame:
        frame_rec = measure_sharded_frame(args, ctx, dev, rank, world, numa_rec)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    k1_traffic, k1_src = ncu_traffic(k1_name)
    k2_traffic, k2_src = ncu_traffic(k2_name)
    mib_rank = nb * BLOCK / 2**20
    ms_per_step = elapsed_ms / args.steps
    value = world * mib_rank / (ms_per_step / 1e3)
    peak, peak_src = measured_peaks()
    alg_bytes = nb * BLOCK + comp_bytes                 # SURVEY.md §8(d): uncompressed + compressed, either direction
    ach_c = alg_bytes / (t_c / 1e3) / 1e9
    ach_d = alg_bytes / (t_d / 1e3) / 1e9

    # CPU baseline on this box's host cores: the whole batch, persistent pool (all cores: undo the NUMA binding first)
    numa.restore_affinity(ninfo)
    if frame_rec is not None:
        frame_rec["cpu_baseline"] = cpu_frame_baseline(8)
    threads, cores = host_topology()
    # the CPU baseline is timed on rank 0 at N=1 only (the other ranks' host pipelines would compete for the cores)
    cpu_all = cpu_arm_fresh_process(nb) if world == 1 else None
    if world == 1 and cpu_all is None:
        cpu_all = dict(cpu_arm(data, nb, threads, 3), how="in this process (the subprocess failed)")
    cpu_one = cpu_arm(data, min(nb, 1024), 1, 2) if world == 1 else None

    line = {
        "metric": METRIC, "value": value, "unit": "MiB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8",
        "data": f"{FIXTURE} tiled (deterministic corpus fixture, BASELINE config 2); inputs larger than L2",
        "config": {"workload": f"{nb} x 64 KiB JSON blocks per GPU (1 GiB), block format, compress+decompress, "
                               f"byte-identical to the oracle", "block_bytes": BLOCK, "blocks_per_gpu": nb,
                   "l2_policy": "inputs (1 GiB in, 0.24 GiB compressed, 1 GiB out per step) larger than the 126 MB L2",
                   "ratio": comp_bytes / (nb * BLOCK)},
        "compress_mibs": world * mib_rank / (t_c / 1e3), "decompress_mibs": world * mib_rank / (t_d / 1e3),
        "compress_ms": t_c, "decompress_ms": t_d,
        # traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture of
        # the same workload (profiles/r1_ncu_summary.json; see ncu_traffic())
        "roofline": {"kernel": k1_name, "bound": "hbm", "achieved": ach_c, "peak": peak,
                     "unit": "GB/s", "frac": ach_c / peak, "traffic": k1_traffic if nb == NBLOCKS_DEFAULT else None,
                     "traffic_source": f"profiles/{k1_src} (ncu --set full capture of this kernel on this workload)" if k1_src else None,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes},
        "roofline_decompress": {"kernel": k2_name, "bound": "hbm", "achieved": ach_d, "peak": peak,
                                "unit": "GB/s", "frac": ach_d / peak,
                                "traffic": k2_traffic if nb == NBLOCKS_DEFAULT else None,
                                "traffic_source": f"profiles/{k2_src}" if k2_src else None, "peak_source": peak_src,
                                "algorithmic_bytes_per_launch": alg_bytes},
        "cpu_baseline": None if cpu_all is None else {
            "value": cpu_all["roundtrip_mibs"], "unit": "MiB/s", "cores": cores, "threads": threads, "kind": "port",
            "sample": f"all {nb} blocks, compress+decompress, {threads} persistent threads on {cores} "
                      f"physical cores (oracle/lz4_cpu_baseline.c: C port of lz4_flex's unsafe path); "
                      + cpu_all.get("how", ""),
            "compress_mibs": cpu_all["compress_mibs"], "decompress_mibs": cpu_all["decompress_mibs"],
            "single_thread": {"compress_mibs": cpu_one["compress_mibs"],
                              "decompress_mibs": cpu_one["decompress_mibs"]},
            "liblz4_anchor": liblz4_anchor(data, min(nb, 1024))},
        # headline = the better of (a) one compress call then one decompress call per step, (b) the stream of batches in which
        # the two calls of consecutive steps share the duplex link; both are in the record, `mode` says which one `value` is
        "e2e": {"value": world * mib_rank / min(e2e_s, stream_s if stream_rec else 1e30), "unit": "MiB/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * min(e2e_s, stream_s if stream_rec else 1e30),
                "mode": "stream of batches" if (stream_rec and stream_s < e2e_s) else "one step at a time",
                "one_step_at_a_time": {"value": world * mib_rank / e2e_s, "ms_per_step": 1e3 * e2e_s},
                "serial_ms_per_step": 1e3 * e2e_serial_s, "chunks": best_chunks, "per_rank": per_rank,
                "compress_call_ms": 1e3 * float(np.mean([c for c, _ in call_t])),
                "decompress_call_ms": 1e3 * float(np.mean([d for _, d in call_t])), "link": link, "stream": stream_rec if stream_rec else ({"error": stream_failed} if stream_failed else None),
                "api": "lz4b200_compress_batch_host + lz4b200_decompress_batch_host (pinned host buffers); "
                       + (stream_rec["how"] if (stream_rec and stream_s < e2e_s) else e2e_how)},
        "gpu_launches": 2 * args.steps,
        "clocks": clocks,
        "numa": numa_rec,
        "sharded_frame": frame_rec,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def hdfs_range(lo: int, n: int) -> np.ndarray:
    """Bytes [lo, lo + n) of hdfs.json tiled by ABSOLUTE offset (BASELINE config 4)."""
    from lz4_flex_b200 import corpus
    src = np.frombuffer(corpus.load("hdfs.json"), dtype=np.uint8)
    i0 = lo % src.size
    reps = -(-(n + i0) // src.size)
    return np.ascontiguousarray(np.tile(src, reps)[i0: i0 + n])


def oracle_frame_from(first_block: int, data: np.ndarray, bs: int) -> bytes:
    """Oracle frame body+header for blocks [first_block, ...) of a 4 MiB-block stream: the reference's persistent table
    driven from the same stream offset (frame/compress.rs:261-371; table epochs per :266-271)."""
    import oracle
    from lz4_flex_b200.frame import BlockSize, FrameInfo
    table = oracle.FrameTable()
    table.offset = first_block * bs
    out = [FrameInfo(block_size=BlockSize.Max4MB).header_bytes()]
    for k in range(0, data.size, bs):
        blk = data[k:k + bs].tobytes()
        c = table.compress(blk, bs)
        out.append(len(c).to_bytes(4, "little") + c if len(c) < len(blk) else (len(blk) | 0x80000000).to_bytes(4, "little") + blk)
    out.append(b"\0\0\0\0")
    return b"".join(out)


def measure_sharded_frame(args, ctx, dev, rank, world, numa_info=None):
    """BASELINE config 4, the multi-GPU path the north star names: ONE LZ4 frame of 4 MiB independent blocks over
    hdfs.json log data tiled by absolute offset, `--frame-blocks` (256) blocks per GPU, block modes by absolute index
    (FRESH at 0, 511, 1022, ...), every rank compresses its contiguous block range and the packed chunks are gathered
    into rank 0's frame buffer INSIDE the timed step (sizes all_gather + pack kernels storing over NVLink + completion
    all_reduce; lz4_flex_b200.sharded.PeerFrameGather).  Returns the record (rank 0) or None."""
    import hashlib
    import torch
    import torch.distributed as dist
    from lz4_flex_b200 import sharded

    bs = 4 << 20
    per = args.frame_blocks
    total = world * per * bs
    mine = hdfs_range(rank * per * bs, per * bs)
    h_in = torch.empty(per * bs, dtype=torch.uint8).pin_memory()
    h_in.numpy()[:] = mine
    d_in = h_in.to(dev, non_blocking=True)

    # ---- parity on a reduced config that crosses the table-epoch boundary: blocks 508.. (6 per rank) vs the oracle ----
    pb = 6
    base = 508
    small = hdfs_range((base + rank * pb) * bs, pb * bs)
    g = sharded.make_frame_gather(world * pb * bs, 7, rank, world, ctx, base_block=base)
    g.step(torch.from_numpy(small).to(dev))
    torch.cuda.synchronize()
    parity = None
    if rank == 0:
        got = g.result().cpu().numpy().tobytes()
        want = oracle_frame_from(base, hdfs_range(base * bs, world * pb * bs), bs)
        parity = {"blocks": world * pb, "first_block": base, "fresh_block_inside": 511,
                  "frame_sha256": hashlib.sha256(got).hexdigest(), "oracle_sha256": hashlib.sha256(want).hexdigest(),
                  "byte_identical_to_oracle": got == want}
    g.close()

    # ---- the timed workload ------------------------------------------------------------------------------------------
    g = sharded.make_frame_gather(total, 7, rank, world, ctx)
    for _ in range(max(args.warmup, 3)):
        g.step(d_in)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    steps = max(1, min(args.steps, 10))
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    kms, xms = [], []
    e0.record()
    for _ in range(steps):
        g.step(d_in, timed=True)
    e1.record()
    torch.cuda.synchronize()
    # per-phase times of the last step (events inside the step); whole-step time from the outer pair
    k_ms, x_ms = g.timings_ms()
    ms = e0.elapsed_time(e1) / steps
    # ---- end to end: host buffer -> H2D -> compress -> gather -> frame on rank 0's host ---------------------------------
    frame_len = int(g.frame_len.item()) if rank == 0 else 0
    h_frame = torch.empty(max(frame_len, 1), dtype=torch.uint8).pin_memory() if rank == 0 else None
    e2e = []
    for it in range(3):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        d_in.copy_(h_in, non_blocking=True)
        g.step(d_in)
        if rank == 0:
            h_frame.copy_(g.result()[:frame_len], non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if it:
            e2e.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e))
    t = torch.tensor([ms, k_ms, x_ms, e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, k_ms, x_ms, e2e_s = [float(v) for v in t.cpu()]
    rec = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        comp_bytes = frame_len
        alg = per * bs + comp_bytes / world                      # per GPU: input read + its share of the frame written
        rec = {
            "workload": f"BASELINE config 4: {world * per} x 4 MiB hdfs.json blocks ({total / 2**30:.0f} GiB), frame format, "
                        f"{per} blocks per GPU, block modes by absolute index, gathered into rank 0's frame buffer",
            "value": total / 2**20 / (ms / 1e3), "unit": "MiB/s", "ms_per_step": ms, "steps": steps,
            "scaling": "weak", "frame_bytes": frame_len, "ratio": frame_len / total,
            "collective": {"compress_kernel_ms": k_ms, "exchange_and_pack_ms": x_ms,
                           "how": "all_gather of the 8-byte packed sizes, then: " + g.transport},
            "roofline": {"kernel": _last_kernel(ctx, 0), "bound": "hbm", "achieved": alg / (k_ms / 1e3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": alg / (k_ms / 1e3) / 1e9 / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg},
            "e2e": {"value": total / 2**20 / e2e_s, "unit": "MiB/s", "ms_per_step": 1e3 * e2e_s,
                    "h2d_bytes_per_step": per * bs, "d2h_bytes_per_step": frame_len,
                    "api": "pinned host range -> H2D -> lz4b200_frame_range_compress -> size exchange -> "
                           "lz4b200_frame_range_pack into rank 0 -> D2H of the frame"},
            "parity": parity, "numa": numa_info,
        }
    g.close()
    return rec


def _last_kernel(ctx, which: int) -> str:
    from lz4_flex_b200 import _native
    return _native.lib().lz4b200_ctx_last_kernel(ctx.handle, which).decode()


def cpu_frame_baseline(nblocks: int):
    """The reference's frame path is ONE thread per frame (FrameEncoder is a single &mut self stream): the CPU port
    compressing `nblocks` 4 MiB hdfs blocks of the frame on one thread."""
    import oracle
    bs = 4 << 20
    data = hdfs_range(0, nblocks * bs)
    t0 = time.perf_counter()
    f = oracle.frame_compress(data, 7)
    dt = time.perf_counter() - t0
    return {"value": nblocks * bs / 2**20 / dt, "unit": "MiB/s", "cores": 1, "kind": "port",
            "sample": f"{nblocks} x 4 MiB blocks of the same stream, one thread (the reference's FrameEncoder is serial per frame)",
            "ratio": len(f) / (nblocks * bs)}


def run_frame(args):
    """--workload frame: only the sharded-frame measurement (the default bench line carries it as `sharded_frame`)."""
    import torch
    import torch.distributed as dist
    from lz4_flex_b200 import block, numa
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ninfo = numa.bind_to_gpu_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = block.Context(local)
    rec = measure_sharded_frame(args, ctx, dev, rank, world, {k: v for k, v in ninfo.items() if k != "original_affinity"})
    if rank == 0:
        numa.restore_affinity(ninfo)
        rec["cpu_baseline"] = cpu_frame_baseline(8)
        rec["n_gpus"] = world
        print(json.dumps(rec))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=NBLOCKS_DEFAULT, help="64 KiB blocks per GPU")
    ap.add_argument("--quick", action="store_true", help="kernel timings only (tuning aid; not a bench line)")
    ap.add_argument("--workload", default="blocks", choices=["blocks", "frame"],
                    help="blocks = BASELINE config 2 (default); frame = config 4 sharded frame + NCCL gather")
    ap.add_argument("--frame-blocks", type=int, default=256, help="4 MiB blocks per GPU for the sharded-frame record")
    ap.add_argument("--no-frame", action="store_true", help="skip the sharded-frame record (tuning aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the block workload computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "blocks"):
        ap.error("--dump-outputs writes the outputs of the GPU block workload (--impl ours --workload blocks)")
    if args.workload == "frame" and args.impl == "ours":
        run_frame(args)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
