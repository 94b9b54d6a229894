#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native LZ4 block codec (see BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

The metric is "GB/s uncompressed (encode+decode) on batched 64 KiB blocks": a STEP is one
L00_FAST encode pass over the configs[2] batch plus one decode pass over the configs[1] batch
(65 536 independent 64 KiB blocks = 4 GiB raw each, per GPU), `value` = uncompressed bytes of both
passes / time.  Inputs are the workload SURVEY.md 8(d) names: the reference's own generator
RDG_genBuffer (orig/programs/datagen.c:156) with matchProba 0.63 (decode, ratio ~0.50) and 0.55
(encode, ratio ~0.57), seed 1234 + chunk index, generated in 64 MiB chunks; both arms build their
inputs with the same code (oracle/: the compiled reference generator, else its checked
restatement) -- only as INPUT DATA, never on a timed path.  With N > 1 every rank owns its own
slice of the block list (weak scaling, the NCCL-free split of configs[4]; NCCL is used only for
the barrier and the max-over-ranks time reduction).

The JSON line carries, beyond the base contract:
  decode / encode  device-timed throughput of each direction (CUDA events around the launches)
  roofline         the decode step (the kernel the north_star target names): algorithmic bytes
                   (compressed read + raw written) / CUDA-event time vs the measured HBM peak;
                   roofline.encode is the same for the encoder (the kernel that dominates the step)
  e2e              the same step through the C-ABI calls with HOST (pinned) buffers: H2D and D2H
                   inside the timed region; e2e.decode / e2e.encode split it
  cpu_baseline     the reference's CPU engine on this box's host cores, bounded sample, median+best
  aux              pickler (configs[3]), and on a multi-GPU box the one-call ALL_DEVICES split

`--impl reference` times the reference's own CPU implementation (oracle/_ref: the upstream C
engine the C# code is a port of and is tested bit-identical against; else the oracle port) with
all host threads on the SAME config; it never loads libk4lz4.
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
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BLOCK = 65536
BLOCKS_PER_GPU = 65536          # configs[1] / configs[2]: 4 GiB of raw data per GPU and direction
BOUND = BLOCK + BLOCK // 255 + 16
MP_DECODE = 0.63                # RDG_genBuffer matchProba: ratio ~0.50 at 64 KiB blocks (configs[1])
MP_ENCODE = 0.55                # ... ratio ~0.57 "Silesia-like" (configs[2])
SEED = 1234
CHUNK_BLOCKS = 1024             # generator streams are 64 MiB long
METRIC = "GB/s uncompressed (encode+decode) on batched 64KiB blocks @1/2/4/8 GPU vs CPU ref"
ALL_CPUS = os.sched_getaffinity(0)     # before any NUMA binding


# ---- pure helpers (unit-tested on CPU, tests/test_host_logic.py) --------------------------------

def shard_range(n_blocks: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous NCCL-free split of the block list: rank r owns [lo, hi)."""
    return n_blocks * rank // world, n_blocks * (rank + 1) // world


def reduce_max_seconds(seconds: float, device="cuda") -> float:
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return seconds
    t = torch.tensor([seconds], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def reduce_sum_int(v: int, device="cuda") -> int:
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return v
    t = torch.tensor([v], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return int(t.item())


def workload_config(blocks_per_gpu: int) -> dict:
    """The `config` object: identical in both arms."""
    return {
        "workload": "batched L00_FAST encode (configs[2]) + decode (configs[1]) of independent 64 KiB blocks, "
                    "LZ4Codec.Encode/Decode semantics, bit-exact",
        "blocks_per_gpu_per_direction": blocks_per_gpu, "block_bytes": BLOCK,
        "generator": "reference datagen RDG_genBuffer(matchProba 0.63 decode / 0.55 encode, litProba 0, "
                     "seed 1234 + chunk) in 64 MiB chunks, cut into 64 KiB blocks",
        "compressed_layout": "decode input tightly packed + int64 offsets; encode output in compressBound slots",
        "l2": "each pass touches > 6 GB >> 126 MB L2; no flush needed",
    }


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic() -> dict | None:
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of every kernel of the step, from the
    committed `ncu --set full` capture of this command (profiles/traffic.json); None if absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None


def gen_blocks(n_blocks: int, match_proba: float, first_block: int, out: np.ndarray | None = None) -> np.ndarray:
    """n_blocks x 64 KiB of the reference generator's output; chunk c = blocks [1024c, 1024c+1024) is
    one RDG_genBuffer stream with seed 1234 + c, so any slice of the global block list is reproducible."""
    import oracle
    eng = oracle.best()
    buf = out if out is not None else np.empty(n_blocks * BLOCK, dtype=np.uint8)
    jobs = []
    b = first_block
    end = first_block + n_blocks
    while b < end:
        c = b // CHUNK_BLOCKS
        hi = min((c + 1) * CHUNK_BLOCKS, end)
        jobs.append((c, b, hi))
        b = hi

    def run(job):
        c, lo, hi = job
        if lo == c * CHUNK_BLOCKS:
            eng.datagen((hi - lo) * BLOCK, match_proba, 0.0, SEED + c,
                        out=buf[(lo - first_block) * BLOCK:(hi - first_block) * BLOCK])
        else:       # slice that starts inside a chunk: generate the chunk prefix, keep the tail
            tmp = eng.datagen((hi - c * CHUNK_BLOCKS) * BLOCK, match_proba, 0.0, SEED + c)
            buf[(lo - first_block) * BLOCK:(hi - first_block) * BLOCK] = tmp[(lo - c * CHUNK_BLOCKS) * BLOCK:]

    with ThreadPoolExecutor(max_workers=min(64, os.cpu_count() or 1)) as ex:
        list(ex.map(run, jobs))
    return buf


DUMP_BLOCKS = 64                # --dump-outputs: blocks whose bytes are written (2 x 16 MiB as float32)


def dump_sample(n_blocks: int) -> np.ndarray:
    """The fixed, seeded sample of block indices whose bytes --dump-outputs writes."""
    return np.sort(np.random.default_rng(SEED).choice(n_blocks, min(DUMP_BLOCKS, n_blocks), replace=False))


def write_outputs(out_dir: str, idx: np.ndarray, enc_len: np.ndarray, enc_slots: np.ndarray,
                  dec_len: np.ndarray, dec_blocks: np.ndarray) -> None:
    """--dump-outputs: what the last timed step returned to its caller, as <out_dir>/<name>.npy -- the
    encode and decode lengths of every block (float64) and, for the blocks `idx`, the compressed bytes
    (one compressBound slot per block, zero past the block's length) and the decoded bytes (float32)."""
    os.makedirs(out_dir, exist_ok=True)
    enc_slots = np.where(np.arange(BOUND)[None, :] < enc_len[idx][:, None], enc_slots, 0)
    for name, a, dt in (("sample_blocks", idx, np.float64), ("encode_lengths", enc_len, np.float64),
                        ("encode_bytes", enc_slots, np.float32), ("decode_lengths", dec_len, np.float64),
                        ("decode_bytes", dec_blocks, np.float32)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a).astype(dt))


def bind_to_gpu_numa_node(index: int) -> str:
    """Pins this process to the CPUs of the NUMA node GPU `index` hangs off (host staging buffers are
    then allocated node-local by first touch).  Best effort; returns a description."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa: single node"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        allowed = ids & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"numa node {node} ({len(allowed)} cpus)"
        return f"numa node {node}: no allowed cpus, unbound"
    except Exception as e:  # noqa: BLE001
        return f"numa: unbound ({type(e).__name__})"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ---- the reference's CPU engine (reference arm, cpu_baseline leg) ---------------------------------

class CpuWorkload:
    """The step on the host: raw_enc --encode--> slots ; comp_dec --decode--> out, `threads` pthreads."""

    def __init__(self, n_blocks: int, first_block: int, threads: int):
        import oracle
        self.eng = oracle.best()
        self.kind = self.eng.kind
        self.nb, self.threads = n_blocks, threads
        self.raw_dec = gen_blocks(n_blocks, MP_DECODE, first_block)
        self.raw_enc = gen_blocks(n_blocks, MP_ENCODE, first_block)
        self.raw_off = np.arange(n_blocks, dtype=np.int64) * BLOCK
        self.raw_len = np.full(n_blocks, BLOCK, dtype=np.int32)
        self.slot_off = np.arange(n_blocks, dtype=np.int64) * BOUND
        self.slot_cap = np.full(n_blocks, BOUND, dtype=np.int32)
        self.slots = np.zeros(n_blocks * BOUND, dtype=np.uint8)
        self.enc_len = np.zeros(n_blocks, dtype=np.int32)
        # decode input: the decode batch compressed once by the same engine (setup, not timed)
        self.comp_dec = np.zeros(n_blocks * BOUND, dtype=np.uint8)
        self.comp_len = np.zeros(n_blocks, dtype=np.int32)
        self.eng.run_batch(0, self.raw_dec, self.raw_off, self.raw_len, self.comp_dec, self.slot_off,
                           self.slot_cap, self.comp_len, threads)
        self.out = np.zeros(n_blocks * BLOCK, dtype=np.uint8)
        self.out_len = np.zeros(n_blocks, dtype=np.int32)
        self.ratio_dec = float(self.comp_len.sum()) / (n_blocks * BLOCK)

    def encode(self) -> float:
        return self.eng.run_batch(0, self.raw_enc, self.raw_off, self.raw_len, self.slots, self.slot_off,
                                  self.slot_cap, self.enc_len, self.threads)

    def decode(self) -> float:
        return self.eng.run_batch(1, self.comp_dec, self.slot_off, self.comp_len, self.out, self.raw_off,
                                  self.raw_len, self.out_len, self.threads)

    def verify(self) -> bool:
        return bool(np.array_equal(self.out, self.raw_dec)) and bool((self.out_len == BLOCK).all()) \
            and bool((self.enc_len > 0).all())

    def time_steps(self, warmup: int, steps: int):
        for _ in range(warmup):
            self.encode(); self.decode()
        te, td = [], []
        for _ in range(steps):
            te.append(self.encode()); td.append(self.decode())
        return te, td


def cpu_numbers(w: CpuWorkload, te: list, td: list) -> dict:
    ub = w.nb * BLOCK
    tot = [a + b for a, b in zip(te, td)]
    return {
        "combined_gbs_mean": 2 * ub * len(tot) / sum(tot) / 1e9,
        "combined_gbs_median": 2 * ub / statistics.median(tot) / 1e9,
        "combined_gbs_best": 2 * ub / min(tot) / 1e9,
        "decode_gbs_median": ub / statistics.median(td) / 1e9, "decode_gbs_best": ub / min(td) / 1e9,
        "encode_gbs_median": ub / statistics.median(te) / 1e9, "encode_gbs_best": ub / min(te) / 1e9,
    }


def engine_name(kind: str) -> str:
    return ("reference upstream C engine orig/lib/lz4.c (oracle/_ref), native-C stand-in for the K4os C# engine "
            "(no .NET runtime in the image)") if kind == "reference" else "oracle port (k4lz4_oracle.c)"


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0)) or 1
    nb = args.blocks
    w = CpuWorkload(nb, 0, threads)
    te, td = w.time_steps(args.warmup, args.steps)
    if args.dump_outputs:
        idx = dump_sample(nb)
        write_outputs(args.dump_outputs, idx, w.enc_len, w.slots.reshape(nb, BOUND)[idx], w.out_len,
                      w.out.reshape(nb, BLOCK)[idx])
    ok = w.verify()
    r = cpu_numbers(w, te, td)
    t = sum(te) + sum(td)
    gbs = r["combined_gbs_mean"]
    sample = (f"the full config: {nb} x 64 KiB blocks per direction per step (decode ratio {w.ratio_dec:.3f}, "
              f"encode ratio {float(w.enc_len.sum()) / (nb * BLOCK):.3f}), {threads} pinned pthreads over contiguous block ranges")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 3), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * t / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(nb),
        "engine": engine_name(w.kind), "verified": ok,
        "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": threads, "kind": w.kind, "sample": sample,
                         **{k: round(v, 3) for k, v in r.items()}},
        "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- our arm ----------------------------------------------------------------------------------------

def all_devices_leg(torch, N, L, h_comp, comp_bytes, h_comp_len, h_raw_enc, nb, h_raw_dec, steps) -> dict:
    """One process, one call per direction, every visible GPU: the block list is `ndev` copies of this
    rank's batch; slice g lives in pinned memory allocated next to GPU g."""
    import ctypes
    ndev = torch.cuda.device_count()
    try:
        os.sched_setaffinity(0, ALL_CPUS)                        # rank 0 was bound to GPU 0's node
    except OSError:
        pass
    comp_sl, out_sl, raw_sl, slot_sl = [None] * ndev, [None] * ndev, [None] * ndev, [None] * ndev

    def alloc(g):
        bind_to_gpu_numa_node(g)                                 # affects only this thread's process mask on Linux
        comp_sl[g] = torch.empty(comp_bytes + 64, dtype=torch.uint8).pin_memory()
        comp_sl[g][:comp_bytes].copy_(h_comp[:comp_bytes])
        out_sl[g] = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
        raw_sl[g] = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
        raw_sl[g].copy_(h_raw_enc)
        slot_sl[g] = torch.empty(nb * BOUND, dtype=torch.uint8).pin_memory()
    ths = [threading.Thread(target=alloc, args=(g,)) for g in range(ndev)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    try:
        os.sched_setaffinity(0, ALL_CPUS)
    except OSError:
        pass
    n = ndev * nb
    base_c = min(t.data_ptr() for t in comp_sl)
    base_o = min(t.data_ptr() for t in out_sl)
    base_r = min(t.data_ptr() for t in raw_sl)
    base_s = min(t.data_ptr() for t in slot_sl)
    rel = np.zeros(nb, dtype=np.int64)
    rel[1:] = np.cumsum(h_comp_len[:-1].astype(np.int64))
    c_off = np.concatenate([rel + (comp_sl[g].data_ptr() - base_c) for g in range(ndev)])
    c_len = np.tile(h_comp_len, ndev).astype(np.int32)
    blk = np.arange(nb, dtype=np.int64)
    o_off = np.concatenate([blk * BLOCK + (out_sl[g].data_ptr() - base_o) for g in range(ndev)])
    r_off = np.concatenate([blk * BLOCK + (raw_sl[g].data_ptr() - base_r) for g in range(ndev)])
    s_off = np.concatenate([blk * BOUND + (slot_sl[g].data_ptr() - base_s) for g in range(ndev)])
    o_cap = np.full(n, BLOCK, dtype=np.int32)
    s_cap = np.full(n, BOUND, dtype=np.int32)
    o_len = np.empty(n, dtype=np.int32)
    e_len = np.empty(n, dtype=np.int32)

    def dec():
        N.check(L.k4lz4_decode_batch(base_c, c_off.ctypes.data, c_len.ctypes.data, base_o, o_off.ctypes.data,
                                     o_cap.ctypes.data, o_len.ctypes.data, n, N.MEM_HOST, None, N.ALL_DEVICES))

    def enc():
        N.check(L.k4lz4_encode_batch(base_r, r_off.ctypes.data, o_cap.ctypes.data, base_s, s_off.ctypes.data,
                                     s_cap.ctypes.data, e_len.ctypes.data, n, 0, N.MEM_HOST, None, N.ALL_DEVICES))
    dec(); enc()
    td = te = 0.0
    for _ in range(steps):
        a = time.perf_counter(); enc(); b = time.perf_counter(); dec(); c = time.perf_counter()
        te += b - a; td += c - b
    ok = bool((o_len == BLOCK).all()) and all(bool(torch.equal(out_sl[g][:BLOCK * 64], h_raw_dec[:BLOCK * 64])) for g in range(ndev)) \
        and bool((e_len.reshape(ndev, nb) == e_len[:nb]).all())
    ub = n * BLOCK
    return {"gpus": ndev, "blocks": n, "verified": ok,
            "decode_gbs": round(ub * steps / td / 1e9, 2), "encode_gbs": round(ub * steps / te / 1e9, 2),
            "combined_gbs": round(2 * ub * steps / (td + te) / 1e9, 2),
            "api": "one k4lz4_encode_batch + one k4lz4_decode_batch call, memKind=HOST, device=K4LZ4_ALL_DEVICES, "
                   "NUMA-local pinned slices"}


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist
    from k4os.compression.lz4_b200 import _native as N, batch as B
    if args.lib:
        N.SO_PATH = os.path.abspath(args.lib)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl ours) needs a CUDA device; there is no CPU fallback")
    numa = bind_to_gpu_numa_node(local) if not args.no_numa else "numa: binding disabled"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")   # host-side waits that keep the GPUs idle (aux leg below)
    L = N.lib()
    nb = args.blocks
    total_blocks = nb * world
    lo, hi = shard_range(total_blocks, rank, world)
    assert hi - lo == nb
    stream = torch.cuda.current_stream().cuda_stream

    def dptr(t):
        return t.data_ptr()

    # ---- inputs: reference generator on the host (pinned), then resident in HBM ----
    h_raw_enc = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
    h_raw_dec = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
    gen_blocks(nb, MP_ENCODE, lo, out=h_raw_enc.numpy())
    gen_blocks(nb, MP_DECODE, lo, out=h_raw_dec.numpy())
    raw_enc = h_raw_enc.to(dev, non_blocking=True)
    raw_dec = h_raw_dec.to(dev, non_blocking=True)
    raw_off = torch.arange(nb, dtype=torch.int64, device=dev) * BLOCK
    raw_len = torch.full((nb,), BLOCK, dtype=torch.int32, device=dev)
    slots = torch.empty(nb * BOUND, dtype=torch.uint8, device=dev)
    slot_off = torch.arange(nb, dtype=torch.int64, device=dev) * BOUND
    slot_cap = torch.full((nb,), BOUND, dtype=torch.int32, device=dev)
    enc_len = torch.empty(nb, dtype=torch.int32, device=dev)
    comp_len = torch.empty(nb, dtype=torch.int32, device=dev)
    # decode input: the decode batch compressed by our own (bit-exact) encoder, tightly packed
    B.encode_batch_device(dptr(raw_dec), dptr(raw_off), dptr(raw_len), dptr(slots), dptr(slot_off),
                          dptr(slot_cap), dptr(comp_len), nb, 0, stream)
    torch.cuda.synchronize()
    assert int(comp_len.min()) > 0
    comp_off = torch.cumsum(comp_len.to(torch.int64), 0) - comp_len.to(torch.int64)
    comp_bytes = int(comp_len.sum())
    comp = torch.empty(comp_bytes + 64, dtype=torch.uint8, device=dev)
    B.copy_blocks_device(dptr(slots), dptr(slot_off), dptr(comp), dptr(comp_off), dptr(comp_len), nb, stream)
    torch.cuda.synchronize()
    out = torch.empty(nb * BLOCK, dtype=torch.uint8, device=dev)
    out_len = torch.empty(nb, dtype=torch.int32, device=dev)
    ratio_dec = comp_bytes / (nb * BLOCK)

    def encode_pass():
        B.encode_batch_device(dptr(raw_enc), dptr(raw_off), dptr(raw_len), dptr(slots), dptr(slot_off),
                              dptr(slot_cap), dptr(enc_len), nb, 0, stream)

    def decode_pass():
        B.decode_batch_device(dptr(comp), dptr(comp_off), dptr(comp_len), dptr(out), dptr(raw_off),
                              dptr(raw_len), dptr(out_len), nb, stream)

    # ---- warm-up, then K timed steps (device-resident inputs) ----
    warm = max(args.warmup, 3)
    for _ in range(warm):
        encode_pass(); decode_pass()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    B.decode_stats(local, reset=True)
    launches0 = L.k4lz4_launch_count()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    for e0, e1, e2 in evs:
        e0.record(); encode_pass(); e1.record(); decode_pass(); e2.record()
    torch.cuda.synchronize()
    launches = L.k4lz4_launch_count() - launches0
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    paths = B.decode_stats(local, reset=True)
    if args.dump_outputs and rank == 0:              # rank 0's slice: blocks [0, nb) of the global list
        idx = dump_sample(nb)
        d_idx = torch.from_numpy(idx).to(dev)
        write_outputs(args.dump_outputs, idx, enc_len.cpu().numpy(), slots.view(nb, BOUND)[d_idx].cpu().numpy(),
                      out_len.cpu().numpy(), out.view(nb, BLOCK)[d_idx].cpu().numpy())
    enc_ms = [e[0].elapsed_time(e[1]) for e in evs]
    dec_ms = [e[1].elapsed_time(e[2]) for e in evs]
    total_s = reduce_max_seconds(evs[0][0].elapsed_time(evs[-1][2]) / 1e3)
    enc_s = reduce_max_seconds(sum(enc_ms) / 1e3)
    dec_s = reduce_max_seconds(sum(dec_ms) / 1e3)
    # verification: decode == its raw input; encode output decodes back to its raw input
    ok = bool(torch.equal(out, raw_dec)) and bool((out_len == BLOCK).all())
    chk = torch.empty(nb * BLOCK, dtype=torch.uint8, device=dev)
    chk_len = torch.empty(nb, dtype=torch.int32, device=dev)
    B.decode_batch_device(dptr(slots), dptr(slot_off), dptr(enc_len), dptr(chk), dptr(raw_off),
                          dptr(raw_len), dptr(chk_len), nb, stream)
    torch.cuda.synchronize()
    ok = ok and bool(torch.equal(chk, raw_enc)) and bool((chk_len == BLOCK).all())
    del chk
    enc_bytes = int(enc_len.sum())
    ratio_enc = enc_bytes / (nb * BLOCK)
    ok_all = reduce_sum_int(int(ok)) == world
    ub = total_blocks * BLOCK                       # uncompressed bytes per direction per step, all ranks
    value = 2 * ub * args.steps / total_s / 1e9
    peak, peak_src = measured_peak_gbs()
    dec_ms_mean, enc_ms_mean = statistics.mean(dec_ms), statistics.mean(enc_ms)
    algo_dec = comp_bytes + nb * BLOCK
    algo_enc = enc_bytes + nb * BLOCK
    ach_dec = algo_dec / (dec_ms_mean / 1e3) / 1e9
    ach_enc = algo_enc / (enc_ms_mean / 1e3) / 1e9
    traffic = profiled_traffic()

    # ---- e2e: the same step through the C ABI with HOST (pinned) buffers ----
    e2e_steps = max(1, min(args.steps, 3))
    h_comp = torch.empty(comp_bytes + 64, dtype=torch.uint8).pin_memory()
    h_comp[:comp_bytes].copy_(comp[:comp_bytes])
    torch.cuda.synchronize()
    h_comp_off = comp_off.cpu().numpy()
    h_comp_len = comp_len.cpu().numpy()
    h_out = torch.empty(nb * BLOCK, dtype=torch.uint8).pin_memory()
    h_slots = torch.empty(nb * BOUND, dtype=torch.uint8).pin_memory()
    h_raw_off = raw_off.cpu().numpy()
    h_raw_len = raw_len.cpu().numpy()
    h_slot_off = slot_off.cpu().numpy()
    h_slot_cap = slot_cap.cpu().numpy()
    h_out_len = np.empty(nb, dtype=np.int32)
    h_enc_len = np.empty(nb, dtype=np.int32)

    def e2e_encode():
        N.check(L.k4lz4_encode_batch(h_raw_enc.data_ptr(), h_raw_off.ctypes.data, h_raw_len.ctypes.data,
                                     h_slots.data_ptr(), h_slot_off.ctypes.data, h_slot_cap.ctypes.data,
                                     h_enc_len.ctypes.data, nb, 0, N.MEM_HOST, None, local))

    def e2e_decode():
        N.check(L.k4lz4_decode_batch(h_comp.data_ptr(), h_comp_off.ctypes.data, h_comp_len.ctypes.data,
                                     h_out.data_ptr(), h_raw_off.ctypes.data, h_raw_len.ctypes.data,
                                     h_out_len.ctypes.data, nb, N.MEM_HOST, None, local))
    e2e_encode(); e2e_decode()      # warm (allocates the library's staging pools)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    te = td = 0.0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        a = time.perf_counter(); e2e_encode(); b = time.perf_counter(); e2e_decode(); c = time.perf_counter()
        te += b - a; td += c - b
    e2e_s = reduce_max_seconds(time.perf_counter() - t0)
    te, td = reduce_max_seconds(te), reduce_max_seconds(td)
    e2e_ok = bool((h_out_len == BLOCK).all()) and bool(np.array_equal(h_enc_len, enc_len.cpu().numpy())) \
        and bool(torch.equal(h_out[:BLOCK * 256], h_raw_dec[:BLOCK * 256])) \
        and bool(torch.equal(h_slots[:int(h_enc_len[0])], slots[:int(h_enc_len[0])].cpu()))
    e2e_gbs = 2 * ub * e2e_steps / e2e_s / 1e9
    e2e = {"value": round(e2e_gbs, 3), "unit": "GB/s",
           "h2d_bytes_per_step": nb * BLOCK + comp_bytes + 2 * nb * 24,
           "d2h_bytes_per_step": enc_bytes + nb * BLOCK + 2 * nb * 4,
           "steps": e2e_steps, "ms_per_step": round(1e3 * e2e_s / e2e_steps, 2), "verified": bool(e2e_ok),
           "decode": {"value": round(ub * e2e_steps / td / 1e9, 3), "ms": round(1e3 * td / e2e_steps, 2)},
           "encode": {"value": round(ub * e2e_steps / te / 1e9, 3), "ms": round(1e3 * te / e2e_steps, 2)},
           "api": "k4lz4_encode_batch + k4lz4_decode_batch (memKind=HOST), pinned host buffers, " + numa}
    del h_out, h_slots

    aux = {}
    # ---- aux: the product's own multi-GPU path -- ONE k4lz4_decode_batch / k4lz4_encode_batch call with
    # K4LZ4_ALL_DEVICES over world x nb blocks (rank 0 only; the other ranks idle at the barrier below).
    # Host buffers are allocated per GPU slice by a thread pinned to that GPU's NUMA node.
    # (the other ranks wait on a gloo barrier: an NCCL barrier would keep a polling kernel on their GPUs)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
    if rank == 0 and args.all_devices and torch.cuda.device_count() > 1:
        try:
            aux["all_devices_one_call"] = all_devices_leg(torch, N, L, h_comp, comp_bytes, h_comp_len, h_raw_enc, nb,
                                                          h_raw_dec, e2e_steps)
        except Exception as e:   # noqa: BLE001
            aux["all_devices_one_call"] = {"error": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.barrier(group=cpu_group)

    # ---- aux: pickler (configs[3]) device-resident throughput ----
    try:
        if args.no_aux:
            raise RuntimeError("skipped (--no-aux)")
        pn = 1 << 20
        prng = np.random.default_rng(42)
        psz = np.where(prng.random(pn) < 0.5, prng.choice([256, 512, 1024, 2048, 4096], pn),
                       prng.integers(256, 4097, pn)).astype(np.int32)
        pofs = np.zeros(pn, dtype=np.int64); pofs[1:] = np.cumsum(psz[:-1], dtype=np.int64)
        ptot = int(psz.sum())
        if ptot > nb * BLOCK:
            raise RuntimeError("batch too small for the pickler aux run")
        d_po, d_pl = torch.from_numpy(pofs).to(dev), torch.from_numpy(psz).to(dev)
        pko = np.zeros(pn, dtype=np.int64); pko[1:] = np.cumsum(psz[:-1].astype(np.int64) + 1)
        d_pko = torch.from_numpy(pko).to(dev)
        pk = torch.empty(ptot + pn + 16, dtype=torch.uint8, device=dev)
        pkl = torch.zeros(pn, dtype=torch.int32, device=dev)

        def p_run():
            B.pickle_batch_device(dptr(raw_enc), dptr(d_po), dptr(d_pl), dptr(pk), dptr(d_pko), dptr(pkl), pn, 0, stream)
        pout = torch.empty(ptot + 16, dtype=torch.uint8, device=dev)
        pol = torch.zeros(pn, dtype=torch.int32, device=dev)

        def u_run():
            B.unpickle_batch_device(dptr(pk), dptr(d_pko), dptr(pkl), dptr(pout), dptr(d_po), dptr(d_pl), dptr(pol), pn, stream)
        res = {}
        for name, fn in (("pickle", p_run), ("unpickle", u_run)):
            fn(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b)
            res[name] = {"Mmsg_per_s": round(pn / ms / 1e3, 2), "GB_per_s": round(ptot / ms / 1e6, 2), "ms": round(ms, 3)}
        res["verified"] = bool(torch.equal(pout[:ptot], raw_enc[:ptot])) and bool((pol == d_pl).all())
        res["messages"] = pn
        res["ratio"] = round(float(pkl.sum()) / ptot, 4)
        aux["pickler_1M_256B_4KiB"] = res
        del pk, pout
    except Exception as e:   # noqa: BLE001
        aux["pickler_1M_256B_4KiB"] = {"error": str(e)}

    # ---- cpu baseline on rank 0 at N = 1: bounded sample of the same step ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:                                        # the rank was bound to its GPU's NUMA node: the CPU leg gets every core
            os.sched_setaffinity(0, ALL_CPUS)
        except OSError:
            pass
        threads = len(os.sched_getaffinity(0)) or 1
        sb = min(16384, nb)
        w = CpuWorkload(sb, lo, threads)
        steps_cpu = 0
        te_c, td_c = [], []
        t0 = time.perf_counter()
        w.encode(); w.decode()
        while time.perf_counter() - t0 < 12.0 or steps_cpu < 3:
            te_c.append(w.encode()); td_c.append(w.decode()); steps_cpu += 1
        r = cpu_numbers(w, te_c, td_c)
        # bit-exactness of the GPU encoder against the reference engine on the same blocks
        g = slots.view(nb, BOUND)[:sb].cpu().numpy()
        gl = enc_len[:sb].cpu().numpy()
        same = bool(np.array_equal(gl, w.enc_len)) and all(
            np.array_equal(g[i, :gl[i]], w.slots[i * BOUND:i * BOUND + gl[i]]) for i in range(0, sb, 37))
        cpu = {"value": round(r["combined_gbs_median"], 3), "unit": "GB/s", "cores": threads, "kind": w.kind,
               "sample": (f"{sb} x 64 KiB blocks per direction (1 GiB + 1 GiB) of the same step, {steps_cpu} passes, "
                          f"median pass; {threads} pinned pthreads"),
               **{k: round(v, 3) for k, v in r.items()}, "verified": w.verify(),
               "gpu_encode_bit_exact_vs_this_engine": same}
        w1 = CpuWorkload(256, lo, 1)
        t1e, t1d = w1.time_steps(1, 3)
        cpu["single_thread_decode_gbs"] = round(256 * BLOCK / min(t1d) / 1e9, 3)
        cpu["single_thread_encode_gbs"] = round(256 * BLOCK / min(t1e) / 1e9, 3)

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm,
            "ms_per_step": round(1e3 * total_s / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(nb),
            "parallelism": f"block-list split x{world} (NCCL-free)", "verified": bool(ok_all),
            "decode": {"value": round(ub * args.steps / dec_s / 1e9, 2), "unit": "GB/s", "ms_per_pass": round(dec_ms_mean, 4),
                       "ratio": round(ratio_dec, 4), "paths": paths},
            "encode": {"value": round(ub * args.steps / enc_s / 1e9, 2), "unit": "GB/s", "ms_per_pass": round(enc_ms_mean, 4),
                       "ratio": round(ratio_enc, 4)},
            "roofline": {"bound": "hbm", "kernel": "k4::decode_tile_kernel (+ its two near-empty follow-up launches): the decode pass",
                         "achieved": round(ach_dec, 1), "peak": peak, "unit": "GB/s", "frac": round(ach_dec / peak, 4),
                         "traffic": (traffic or {}).get("decode_bytes_per_launch"),
                         "traffic_split": (traffic or {}).get("decode_split"),
                         "algorithmic_bytes_per_launch": algo_dec, "kernel_ms": round(dec_ms_mean, 4),
                         "read_only_frac": round(comp_bytes / (dec_ms_mean / 1e3) / 1e9 / peak, 4),
                         "peak_source": peak_src,
                         "step_share": {"decode": round(sum(dec_ms) / (sum(dec_ms) + sum(enc_ms)), 4),
                                        "encode": round(sum(enc_ms) / (sum(dec_ms) + sum(enc_ms)), 4)},
                         "encode": {"kernel": "k4::encode kernel: the encode pass (dominates the step by time)",
                                    "achieved": round(ach_enc, 1), "frac": round(ach_enc / peak, 4),
                                    "traffic": (traffic or {}).get("encode_bytes_per_launch"),
                                    "algorithmic_bytes_per_launch": algo_enc, "kernel_ms": round(enc_ms_mean, 4)}},
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "cpu_baseline": cpu,
            "aux": aux,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok_all:
        raise SystemExit("verification FAILED")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--blocks", type=int, default=BLOCKS_PER_GPU, help="blocks per GPU and direction (default: configs[1]/[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-all-devices", dest="all_devices", action="store_false",
                    help="skip aux.all_devices_one_call (ONE host-memory call per direction over every visible GPU; "
                         "runs on rank 0 whenever more than one GPU is visible)")
    ap.add_argument("--lib", default=None, help="development only: another build of libk4lz4.so (A/B runs of kernel variants)")
    ap.add_argument("--no-aux", action="store_true", help="development only: skip the aux legs (pickler, all-devices call)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                         "(lengths of every block, bytes of a fixed sample of blocks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
