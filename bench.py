#!/usr/bin/env python
"""bench.py -- GB/s SHA-256-digested on a 100 GB synthetic blob (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's digests as DIR/*.npy

A "step" is one full digest of the blob: leaf SHA-256 over every 16 KiB of blob bytes, the tree levels above them up
to the 8 MiB chunk-digest list, the levels above that, and the root (modelx.tree.v1, DESIGN.md section 3 -- a NEW
chunked identity; the reference's whole-file digest is one serial chain and cannot use a GPU, see `compat` below).

  value    whole-job GB/s with the blob already resident in HBM (CUDA-event timed, max over ranks)
  e2e      the same digest of the same bytes starting from a FILE (tmpfs, page-cache resident -- the form modelx has a
           blob in): every rank streams its chunk range through the library's pinned ring, so file reads, the host
           staging copy, the H2D copies and the D2H of the chunk list + root are all inside the timed region
  e2e_pinned_ceiling   a sample of the blob held in caller-pinned memory (zero-copy H2D): the PCIe ceiling
  compat   the reference-identical whole-file digests (push.go:149-161) of BASELINE configs 3 (32 x 0.5 GB shards)
           and 5 (1000 x 128 MB blobs) through the coalescing digest service, from files, next to the reference's
           3-goroutine CPU path on a sample of the same files
  N > 1    strong scaling: the blob is sharded by chunk index (rank r owns a contiguous chunk range); no collective on
           the hash path, one NCCL all-gather of the 32-byte chunk digests, then every rank finishes the upper levels.

Only the cpu_baseline / compat cpu legs / --impl reference touch oracle/ (the CPU checker); the timed GPU legs call
libmodelxdigest.so through modelx_b200.  The reference arm never loads libmodelxdigest.so.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import ctypes
import json
import mmap
import os
import shutil
import statistics
import struct
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0x6D6F64656C78  # "modelx"
GB = 1e9


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=float, default=100e9, help="blob bytes (default: the 100 GB metric blob)")
    ap.add_argument("--chunk", type=int, default=8 << 20)
    ap.add_argument("--leaf", type=int, default=16 << 10)
    ap.add_argument("--fanout", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-compat", action="store_true")
    ap.add_argument("--cpu-sample-gb", type=float, default=16.0)
    ap.add_argument("--ref-sample-gb", type=float, default=4.0)
    ap.add_argument("--pinned-gb", type=float, default=16.0, help="pinned-memory sample for e2e_pinned_ceiling")
    ap.add_argument("--compat5-blobs", type=int, default=1000)
    ap.add_argument("--compat5-blob-mb", type=float, default=128.0)
    ap.add_argument("--compat3-shards", type=int, default=32)
    ap.add_argument("--compat3-shard-gb", type=float, default=0.5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the chunk digests and the root of the last timed step to DIR/<name>.npy (float32), so "
                         "that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1")
    return args


def dump_outputs(d, chunk_list: bytes, root: bytes):
    """The digests a caller of the timed path receives, one byte per float32 element (exact for 0..255): the
    32-byte chunk digests as an (nchunks, 32) array and the 32-byte root.  The 100 GB blob has 11,921 chunks, 1.5 MB."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "chunk_digests.npy"), np.frombuffer(chunk_list, dtype=np.uint8).reshape(-1, 32).astype(np.float32))
    np.save(os.path.join(d, "root.npy"), np.frombuffer(root, dtype=np.uint8).astype(np.float32))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """DRAM bytes per algorithmic byte of the leaf kernel from the committed ncu capture (or None)."""
    p = os.path.join(ROOT, "profiles", "ncu_leaf_kernel.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


def host_cpu_info():
    """What the process may actually use: a 128-CPU box with a cgroup quota of 16 CPUs has 16 (VERDICT r1 weak 10)."""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        info["affinity"] = None
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(p) as f:
                info["cgroup_" + os.path.basename(p)] = f.read().strip()
        except OSError:
            pass
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    info["model"] = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    quota = None
    cm = info.get("cgroup_cpu.max", "")
    if cm and cm.split()[0] != "max":
        try:
            quota = float(cm.split()[0]) / float(cm.split()[1])
        except (ValueError, IndexError, ZeroDivisionError):
            quota = None
    info["cgroup_cpus"] = quota
    usable = info["affinity"] or info["os_cpu_count"] or 1
    if quota:
        usable = max(1, min(usable, int(quota)))
    info["usable_threads"] = usable
    return info


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, power, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [c for c, p in zip(sm, power) if p > 250] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def shm_dir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()


# ==================================================================================================
# reference arm: the reference's own CPU implementation of the path, restated in oracle/ (the Go
# toolchain is absent, see DESIGN.md).  Client.digest (pkg/client/push.go:149-161): one goroutine,
# one serial SHA-256 chain over the whole file through a 32 KiB read loop.
# ==================================================================================================
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests.oracle_lib import Oracle
    orc = Oracle()
    nbytes = int(args.ref_sample_gb * (1 << 30))
    path = os.path.join(shm_dir(), f"modelx_b200_ref_sample_{os.getpid()}.bin")
    piece = 256 << 20
    buf = ctypes.create_string_buffer(piece)
    with open(path, "wb") as f:                      # untimed: materialise the sample of the metric blob
        off = 0
        while off < nbytes:
            n = min(piece, nbytes - off)
            orc.gen_into(ctypes.addressof(buf), off, n, SEED)
            f.write(buf.raw[:n] if n < piece else buf.raw)
            off += n
    try:
        for _ in range(args.warmup):
            orc.client_digest(path)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            d, size = orc.client_digest(path)
        dt = time.perf_counter() - t0
    finally:
        os.unlink(path)
    val = nbytes * args.steps / dt / GB
    sample = (f"first {args.ref_sample_gb:g} GiB of the {args.size/1e9:g} GB metric blob as a tmpfs file per step; "
              "Client.digest = 32 KiB read loop + SHA-256 (SHA-NI), one thread: a blob is one serial chain, "
              "the reference cannot use more cores for it (its 3 goroutines hash 3 different blobs, push.go:27)")
    line = {
        "impl": "reference", "metric": "GB/s SHA-256-digested on 100 GB synthetic blob", "value": val, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"{args.size/1e9:g} GB blob, whole-file sha256 (reference semantics, push.go:149-161)",
                   "blob_bytes": int(args.size), "sample_bytes": nbytes},
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": 1, "kind": "port", "sample": sample,
                         "engine": "sha-ni" if orc.engine() == 1 else "portable", "host": host_cpu_info()},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "digest": orc.digest_string(d),
        "native_so_loaded": "libmodelxdigest" in open("/proc/self/maps").read(),   # must be False: the product is not in this process
    }
    print(json.dumps(line), flush=True)


# ==================================================================================================
# helpers of this repo's arm
# ==================================================================================================
def gpu_local_cpus(gpu_index: int):
    """CPUs on the NUMA node the GPU hangs off (sysfs local_cpulist of its PCI function), or None."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out          # "00000000:1b:00.0" -> "0000:1b:00.0"
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        return (cpus & allowed) or None
    except (OSError, ValueError, subprocess.SubprocessError):
        return None


def write_device_range_to_file(torch, blob, nbytes, path, file_offset, threads=8, cpus=None):
    """Untimed setup: device bytes -> file (pinned bounce buffer, parallel pwrite).  With `cpus` the writer threads run on
    those CPUs, so the page cache pages of this range are first-touched on that NUMA node."""
    old = os.sched_getaffinity(0)
    if cpus:
        os.sched_setaffinity(0, cpus)        # threads created below inherit it
    try:
        _write_device_range_to_file(torch, blob, nbytes, path, file_offset, threads)
    finally:
        if cpus:
            os.sched_setaffinity(0, old)


def _write_device_range_to_file(torch, blob, nbytes, path, file_offset, threads):
    piece = 512 << 20
    host = torch.empty(piece, dtype=torch.uint8, pin_memory=True)
    fd = os.open(path, os.O_WRONLY)
    try:
        with cf.ThreadPoolExecutor(threads) as ex:
            off = 0
            while off < nbytes:
                n = min(piece, nbytes - off)
                host[:n].copy_(blob[off:off + n])
                torch.cuda.synchronize()
                mv = memoryview(host.numpy())[:n]
                sub = -(-n // threads)
                futs = [ex.submit(os.pwrite, fd, mv[s:min(s + sub, n)], file_offset + off + s) for s in range(0, n, sub)]
                for fu in futs:
                    fu.result()
                off += n
    finally:
        os.close(fd)


def safetensors_header(payload_bytes: int, shard_index: int) -> bytes:
    """An 8-byte LE header length + JSON header in the safetensors layout, naming fp16 tensors of Llama-3-8B decoder
    layers (q/k/v/o/gate/up/down + norms) that tile `payload_bytes` (the last tensor takes the remainder)."""
    shapes = [("self_attn.q_proj.weight", (4096, 4096)), ("self_attn.k_proj.weight", (1024, 4096)),
              ("self_attn.v_proj.weight", (1024, 4096)), ("self_attn.o_proj.weight", (4096, 4096)),
              ("mlp.gate_proj.weight", (14336, 4096)), ("mlp.up_proj.weight", (14336, 4096)),
              ("mlp.down_proj.weight", (4096, 14336)), ("input_layernorm.weight", (4096,)),
              ("post_attention_layernorm.weight", (4096,))]
    hdr, off, layer = {"__metadata__": {"format": "pt"}}, 0, shard_index
    while off < payload_bytes:
        for name, shape in shapes:
            n = 2
            for s in shape:
                n *= s
            if off + n > payload_bytes:
                n = payload_bytes - off
                shape = (n // 2,)
            if n <= 0:
                break
            hdr[f"model.layers.{layer}.{name}"] = {"dtype": "F16", "shape": list(shape), "data_offsets": [off, off + n]}
            off += n
        layer += 1
    js = json.dumps(hdr, separators=(",", ":")).encode()
    js += b" " * (-len(js) % 8)
    return struct.pack("<Q", len(js)) + js


def cpu_ref3(orc, paths):
    """The reference's blob fan-out: PullPushConcurrency = 3 goroutines, each Client.digest on one file (push.go:27,34-52)."""
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(3) as ex:
        res = list(ex.map(orc.client_digest, paths))
    return time.perf_counter() - t0, res


# ==================================================================================================
# this repo's arm
# ==================================================================================================
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import modelx_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    run_tag = os.environ.get("MASTER_PORT", str(os.getpid())) if world > 1 else str(os.getpid())

    size = int(args.size)
    tp = (args.chunk, args.leaf, args.fanout)
    from modelx_b200 import shard
    nchunks = shard.chunk_count(size, args.chunk)
    per = shard.chunks_per_rank(nchunks, world)      # chunks per rank (only tail ranks may own fewer)
    c0, c1 = shard.chunk_range(rank, world, nchunks)
    b0, b1 = shard.byte_range(rank, world, size, args.chunk)
    my_bytes = b1 - b0
    my_chunks = c1 - c0

    eng = modelx_b200.Engine(devices=[local])
    stream = torch.cuda.current_stream().cuda_stream
    fill = max((my_bytes + 7) // 8 * 8, 8)
    blob = torch.empty(fill, dtype=torch.uint8, device=dev)
    eng.dev_gen_fill(0, blob.data_ptr(), b0, fill, SEED, stream)   # bytes [b0, b1) of the one logical blob
    d_local = torch.zeros(per * 32, dtype=torch.uint8, device=dev)
    d_all = torch.zeros(world * per * 32, dtype=torch.uint8, device=dev)
    d_root = torch.zeros(32, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(xs):
        t = torch.tensor(list(xs), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def step():
        if my_bytes or world == 1:
            eng.dev_tree_chunks(0, blob.data_ptr(), my_bytes, tp, d_local.data_ptr(), stream)
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_local)       # 32 B per chunk; the only exchange on the path
            eng.dev_tree_finish(0, d_all.data_ptr(), nchunks, size, tp, d_root.data_ptr(), stream)
        else:
            eng.dev_tree_finish(0, d_local.data_ptr(), nchunks, size, tp, d_root.data_ptr(), stream)

    # ---- kernel-only: blob resident in HBM ----------------------------------------------------
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.prof_enable(True)
    st0 = eng.stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    prof = eng.prof_read()
    eng.prof_enable(False)
    st1 = eng.stats()
    clocks = sampler.stop() if rank == 0 else None
    ms_max = max_over_ranks(ms)
    value = size * args.steps / (ms_max * 1e-3) / GB
    root_dev = bytes(d_root.cpu().numpy().tobytes())
    chunk_list_dev = bytes((d_all if world > 1 else d_local).cpu().numpy().tobytes())[:nchunks * 32]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, chunk_list_dev, root_dev)
    launches = st1["kernel_launches"] - st0["kernel_launches"]

    # roofline of the dominant kernel: the leaf-level launch (reads every blob byte once)
    peak, peak_src = load_peaks()
    leaf_ms = prof["kernel_ms"] / max(prof["launches"], 1)
    leaf_bytes = prof["bytes"] / max(prof["launches"], 1)
    achieved = leaf_bytes / (leaf_ms * 1e-3) / GB if leaf_ms > 0 else 0.0
    tr = load_traffic()
    # the bound that actually binds: ALU-pipe issue (2 warp-instr/clk/SM measured; 1,056 ALU-pipe instructions per
    # 64-byte block of 32 lanes: 672 SHF + 352 LOP3 + 16 PRMT + 16 loop/address) at the SM clock seen under load
    props = torch.cuda.get_device_properties(dev)
    sm_clk_hz = (clocks["sm_mhz"] if (clocks and clocks.get("sm_mhz")) else 1965.0) * 1e6
    alu_ceiling = 4 * 32 * 64 / (1056 * 2.0) * props.multi_processor_count * sm_clk_hz / GB
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (tr["dram_bytes_per_algorithmic_byte"] * leaf_bytes) if tr else None,
                "kernel": tr.get("kernel", "k_tree_leaves (leaf level)") if tr else "k_tree_leaves (leaf level)",
                "kernel_ms_per_launch": leaf_ms,
                "algorithmic_bytes_per_launch": leaf_bytes, "kernel_share_of_step": prof["kernel_ms"] / ms if ms else None,
                "peak_source": peak_src,
                "alu_pipe": {"ceiling": alu_ceiling, "unit": "GB/s", "frac": achieved / alu_ceiling if alu_ceiling else None,
                             "how": "4 SMSP x 32 lanes x 64 B / (1056 ALU-pipe instr x 2 clk) x SMs x SM clock; pipe rates "
                                    "measured in profiles/r01_pipes_ubench.txt, r02_halfwarp_ubench.txt"},
                "note": ("SHA-256 is 1 B read per B digested but ~16.5 INT32 ALU-pipe instructions per byte; the binding "
                         "limit is the ALU pipe (2 warp-instr/clk/SM measured), ceiling ~1.13 TB/s = 17% of HBM peak; "
                         "see DESIGN.md section 5")}

    # ---- end to end from a FILE: what modelx has (a blob on disk), through the pinned ring --------------------------
    e2e = e2e_pinned = None
    blob_path = os.path.join(shm_dir(), f"modelx_b200_bench_{run_tag}.bin")
    file_bytes = 0
    notes = []
    if not args.no_e2e:
        free = shutil.disk_usage(shm_dir()).free
        file_bytes = size if free > size * 1.05 + (8 << 30) else 0
        if not file_bytes:
            notes.append(f"{shm_dir()} has {free/1e9:.0f} GB free: the {size/1e9:g} GB blob does not fit, e2e from a file skipped")
    if file_bytes:
        t_file = time.perf_counter()
        if rank == 0:
            with open(blob_path, "wb") as f:
                f.truncate(size)
        barrier()
        if my_bytes:
            write_device_range_to_file(torch, blob, my_bytes, blob_path, b0, cpus=gpu_local_cpus(local))
        barrier()
        t_file = time.perf_counter() - t_file

        def e2e_step():
            mine = eng.tree_chunks_file(blob_path, b0, my_bytes, *tp)[:my_chunks * 32] if (my_bytes or world == 1) else b""
            if world > 1:
                d_local.zero_()
                if mine:
                    d_local[:len(mine)].copy_(torch.frombuffer(bytearray(mine), dtype=torch.uint8))
                dist.all_gather_into_tensor(d_all, d_local)
                allc = bytes(d_all.cpu().numpy().tobytes())[:nchunks * 32]
            else:
                allc = mine
            return allc, eng.tree_finish(allc, size, *tp)

        e2e_warm = min(args.warmup, 3)
        for _ in range(e2e_warm):
            e2e_step()
        barrier()
        s0 = eng.stats()
        eng.prof_enable(True)            # device time of the leaf launches inside the e2e region (overlap evidence)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            allc, root_e2e = e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        s1 = eng.stats()
        prof_e2e = eng.prof_read()
        eng.prof_enable(False)
        barrier()
        dt_max = max_over_ranks(dt)
        hb = sum_over_ranks([s1["h2d_bytes"] - s0["h2d_bytes"], s1["d2h_bytes"] - s0["d2h_bytes"],
                             s1["src_bytes_read"] - s0["src_bytes_read"]])
        if root_e2e != root_dev or allc != chunk_list_dev:
            raise SystemExit("e2e digest differs from the HBM-resident digest of the same bytes")
        e2e = {"value": size * args.steps / dt_max / GB, "unit": "GB/s",
               "h2d_bytes_per_step": int(hb[0] / args.steps), "d2h_bytes_per_step": int(hb[1] / args.steps),
               "file_bytes_read_per_step": int(hb[2] / args.steps),
               "ms_per_step": dt_max / args.steps * 1e3, "warmup": e2e_warm,
               "leaf_kernel_ms_per_step": prof_e2e["kernel_ms"] / args.steps, "leaf_launches_per_step": prof_e2e["launches"] / args.steps,
               "source": f"file on tmpfs ({shm_dir()}, page-cache resident, {size/1e9:g} GB, written in {t_file:.1f} s of untimed setup, each rank's "
                         "range first-touched on its GPU's NUMA node); "
                         "each rank preads its chunk range into the library's pinned ring (4 x 64 MiB slots, filler threads bound "
                         "to the GPU's NUMA node), H2D on a copy stream, leaf kernels on a compute stream",
               "api": "mxd_tree_chunks_file(path, rank's byte range) [+ NCCL all-gather of 32 B/chunk] + mxd_tree_finish",
               "overlap": "leaf-kernel device time per step (leaf_kernel_ms_per_step) is hidden behind the copies; slot timeline "
                          "in profiles/r02_e2e_slot_timeline.txt",
               "host_bound": {"usable_cpus": host_cpu_info()["usable_threads"], "ranks_on_this_node": world,
                              "note": "staging a page-cache file into the pinned ring costs one CPU copy per byte (~3 GB/s per core); "
                                      "the ranks of a node share the CPUs the container may use (cgroup quota), so beyond "
                                      "usable_cpus/16 ranks e2e is bound by host cores, not by PCIe or the GPUs -- compare "
                                      "e2e_pinned_ceiling, which scales with the GPUs"}}

    # ---- PCIe ceiling: a sample of the blob in caller-pinned memory (zero-copy H2D, no staging copy) ------------------
    host_ptr = 0
    pin_bytes = int(min(args.pinned_gb * 1e9, my_bytes)) // args.chunk * args.chunk
    if not args.no_e2e and pin_bytes:
        t_pin = time.perf_counter()
        host_ptr = eng.host_alloc(pin_bytes)
        t_pin = time.perf_counter() - t_pin
        host_np = np.frombuffer((ctypes.c_uint8 * pin_bytes).from_address(host_ptr), dtype=np.uint8)
        torch.from_numpy(host_np).copy_(blob[:pin_bytes])
        torch.cuda.synchronize()
        want = None
        for _ in range(2):
            want = eng.tree_chunks_ptr(host_ptr, pin_bytes, *tp)
        barrier()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            got = eng.tree_chunks_ptr(host_ptr, pin_bytes, *tp)
        dtp = max_over_ranks((time.perf_counter() - t0) / reps)
        if got != want or got[:32] != chunk_list_dev[c0 * 32:c0 * 32 + 32]:
            raise SystemExit("pinned-memory digest differs from the HBM-resident digest of the same bytes")
        e2e_pinned = {"value": world * pin_bytes / dtp / GB, "unit": "GB/s", "bytes_per_rank": pin_bytes,
                      "what": f"first {pin_bytes/1e9:.1f} GB of each rank's range held in caller-pinned memory (mxd_host_alloc; pinning "
                              f"took {t_pin:.1f} s = {pin_bytes/1e9/max(t_pin,1e-9):.1f} GB/s and is NOT in this figure): the copy engine "
                              "reads the caller's pages directly, so this is the PCIe Gen5 x16 ceiling for e2e, not a path modelx has"}
        eng.host_free(host_ptr)
        host_ptr = 0
    del blob
    torch.cuda.empty_cache()

    # ---- compat: the reference-identical whole-file digests of BASELINE configs 3 and 5, from files ----------------
    compat = None
    if not args.no_compat:
        try:
            compat = run_compat(args, eng, torch, dist, dev, world, rank, run_tag, barrier, max_over_ranks, sum_over_ranks)
        except Exception as e:   # the headline must still print
            compat = {"error": f"{type(e).__name__}: {e}"}

    # ---- CPU baseline on rank 0's host cores (N=1 only): oracle port, bounded sample ------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and file_bytes:
        from tests.oracle_lib import Oracle
        orc = Oracle()
        host = host_cpu_info()
        with open(blob_path, "rb") as f:
            mm = mmap.mmap(f.fileno(), 0, prot=mmap.PROT_READ)
        try:
            arr = np.frombuffer(mm, dtype=np.uint8)
            base = arr.ctypes.data
            sample = int(min(args.cpu_sample_gb * 1e9, size))
            t0 = time.perf_counter()
            orc.sha256_ptr(base, sample)                               # reference semantics: one serial chain, 1 thread
            dt1 = time.perf_counter() - t0
            t0 = time.perf_counter()                                   # the reference's PullPushConcurrency = 3 (push.go:27)
            orc.tree_digest_ptr(base, sample, *tp, threads=3)
            dt3 = time.perf_counter() - t0
            scaling = {}
            threads = host["usable_threads"]
            for th in sorted({8, 16, 32, 64, threads}):
                if th > (host["affinity"] or th):
                    continue
                t0 = time.perf_counter()
                orc.tree_digest_ptr(base, sample, *tp, threads=th)
                scaling[str(th)] = sample / (time.perf_counter() - t0) / GB
            best_threads = int(max(scaling, key=scaling.get)) if scaling else threads
            t0 = time.perf_counter()
            want_chunks, _, want_root = orc.tree_digest_ptr(base, size, *tp, threads=best_threads)
            dtn = time.perf_counter() - t0
            parity = (want_root == root_dev and b"".join(want_chunks) == chunk_list_dev)
            if not parity:
                raise SystemExit("GPU tree digest differs from the CPU oracle on the full blob")
            del arr
            cpu = {"value": sample / dt1 / GB, "unit": "GB/s", "cores": 1, "kind": "port",
                   "sample": f"first {sample/1e9:g} GB of the blob, one SHA-256 chain on one thread (what the reference does "
                             "for one blob, push.go:149-161), SHA-NI, data already in memory (no read syscalls)",
                   "engine": "sha-ni" if orc.engine() == 1 else "portable", "host": host,
                   "three_threads_tree": {"value": sample / dt3 / GB, "unit": "GB/s", "cores": 3,
                                          "sample": f"first {sample/1e9:g} GB, tree digest on 3 threads (the reference's PullPushConcurrency)"},
                   "all_cores_tree": {"value": size / dtn / GB, "unit": "GB/s", "cores": best_threads,
                                      "sample": "the whole blob (mmap of the same tmpfs file), the same tree digest chunk-parallel on "
                                                "host threads; thread count = the best of the sweep below",
                                      "thread_sweep_gbs": scaling, "parity_with_gpu": parity}}
        finally:
            try:
                mm.close()
            except BufferError:
                pass
    if rank == 0 and os.path.exists(blob_path):
        os.unlink(blob_path)

    if rank == 0:
        like = None
        if cpu and e2e:
            like = {"what": "the SAME digest (modelx.tree.v1) on the same bytes, GPU vs every usable host core",
                    "e2e_file_over_cpu_all_cores_tree": e2e["value"] / cpu["all_cores_tree"]["value"],
                    "hbm_resident_over_cpu_all_cores_tree": value / cpu["all_cores_tree"]["value"],
                    "note": "the reference arm (--impl reference) is the reference's OWN digest: one whole-file SHA-256 chain on one "
                            "core; the ratio against it compares a new chunked identity with the old serial one (DESIGN.md section 3)"}
        line = {
            "metric": "GB/s SHA-256-digested on 100 GB synthetic blob", "value": value, "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{size/1e9:g} GB blob (splitmix64 counter stream) resident in HBM, modelx.tree.v1 digest",
                       "blob_bytes": size, "chunk": args.chunk, "leaf": args.leaf, "fanout": args.fanout,
                       "chunks": nchunks, "parallelism": f"chunk-range sharding x{world}" if world > 1 else "single GPU",
                       "l2": "input per GPU >> 126 MB L2, read once per step (no flush needed)"},
            "clocks": clocks, "e2e": e2e, "e2e_pinned_ceiling": e2e_pinned, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "compat": compat, "like_for_like": like, "notes": notes,
            "root": modelx_b200.digest_string(root_dev),
        }
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_compat(args, eng, torch, dist, dev, world, rank, run_tag, barrier, max_over_ranks, sum_over_ranks):
    """Reference-identical whole-file SHA-256 (push.go:149-161 / pull.go:115-123) of many files at once, from files,
    through the coalescing digest service; files are dealt round-robin over the ranks (no collective)."""
    import modelx_b200
    d = os.path.join(shm_dir(), f"modelx_b200_compat_{run_tag}_{rank}")
    os.makedirs(d, exist_ok=True)
    out = {"identity": "whole-file SHA-256, bit-identical to the reference's Descriptor.Digest",
           "note": "one file = one serial SHA-256 chain (~0.08 GB/s on the GPU); throughput comes only from the number of "
                   "files in flight, so config 3 (32 chains) is slower than three SHA-NI cores and config 5 (1000 chains) is faster; "
                   "adding GPUs adds PCIe lanes and SM sub-partitions but not chains (DESIGN.md section 6)"}
    from tests.oracle_lib import Oracle
    orc = Oracle() if rank == 0 else None
    try:
        # ---------------- config 1: one 64 MB random blob, digest + PutBlob into an in-process registry (rank 0) --------
        if rank == 0:
            from modelx_b200.client import Client, LocalRegistry
            m1 = os.path.join(d, "c1_model")
            os.makedirs(m1)
            with open(os.path.join(m1, "modelx.yaml"), "w") as f:
                f.write("description: bench config 1\n")
            with open(os.path.join(m1, "blob.bin"), "wb") as f:
                f.write(os.urandom(64_000_000))
            cl = Client(eng)
            times = {}
            for mode in ("whole_file", "tree_keyed"):
                best = None
                for rep in range(3):
                    reg = LocalRegistry(os.path.join(d, f"c1_reg_{mode}_{rep}"), eng)
                    t0 = time.perf_counter()
                    (cl.push if mode == "whole_file" else cl.push_tree)(reg, "library/c1", "v1", m1)
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                times[mode] = best
            t0 = time.perf_counter()
            dg, _sz = orc.client_digest(os.path.join(m1, "blob.bin"))
            shutil.copyfile(os.path.join(m1, "blob.bin"), os.path.join(d, "c1_copy.bin"))
            tcpu = time.perf_counter() - t0
            out["config1"] = {"workload": "one 64 MB random blob: digest + PutBlob into the in-process FS registry (+ manifest, index.json)",
                              "gpu_whole_file_identity_ms": times["whole_file"] * 1e3, "gpu_tree_identity_ms": times["tree_keyed"] * 1e3,
                              "cpu_reference_ms": tcpu * 1e3,
                              "note": f"one blob = one serial chain: the reference-identical push is {times['whole_file'] / tcpu:.0f}x slower on the GPU than the reference's "
                                      "CPU digest + copy (mxd_batch_pays_off = false: the Go shim keeps it on the CPU); the tree-keyed push of the "
                                      "same blob reads it once and is bound by the store write"}
            shutil.rmtree(m1, ignore_errors=True)
        # ---------------- config 3: 32 x 0.5 GB safetensors-shaped shards ------------------------------------------------
        nsh, shb = args.compat3_shards, int(args.compat3_shard_gb * 1e9)
        mine = [i for i in range(nsh) if i % world == rank]
        paths = []
        gen = torch.empty(max(shb, 8) // 8 * 8 + 8, dtype=torch.uint8, device=dev)
        for i in mine:
            p = os.path.join(d, f"model-{i + 1:05d}-of-{nsh:05d}.safetensors")
            hdr = safetensors_header(shb - 4096, i) if shb > 8192 else b""
            hdr = hdr[:max(0, shb - 8)]
            payload = shb - len(hdr)
            eng.dev_gen_fill(0, gen.data_ptr(), (i * shb) // 8 * 8, (payload + 7) // 8 * 8, SEED + 3, torch.cuda.current_stream().cuda_stream)
            with open(p, "wb") as f:
                f.write(hdr)
                f.truncate(shb)
            write_device_range_to_file(torch, gen, payload, p, len(hdr))
            paths.append(p)
        barrier()
        for _ in range(1):
            eng.sha256_files(paths) if paths else None
        barrier()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            got, _sizes = eng.sha256_files(paths) if paths else ([], [])
        dt = max_over_ranks((time.perf_counter() - t0) / reps)
        c3 = {"workload": f"{nsh} x {shb/1e9:g} GB safetensors-shaped shards (Llama-3-8B fp16 layout), files on tmpfs",
              "gpu": {"value": nsh * shb / dt / GB, "unit": "GB/s", "ms": dt * 1e3, "files_per_rank": len(mine),
                      "api": "mxd_sha256_files (one coalesced batch per rank)"}}
        if rank == 0 and paths:
            sample = paths[:6]
            tcpu, res = cpu_ref3(orc, sample)
            for (dg, _sz), g in zip(res, got[:len(sample)]):
                if dg != g:
                    raise SystemExit("compat config 3: GPU digest differs from the reference path on the same file")
            c3["cpu_ref_3"] = {"value": len(sample) * shb / tcpu / GB, "unit": "GB/s", "cores": 3,
                               "sample": f"{len(sample)} of the same files, Client.digest (32 KiB read loop, SHA-NI) on 3 threads "
                                         "= PullPushConcurrency; digests compared with the GPU's"}
            c3["pays_off"] = bool(modelx_b200.batch_pays_off(nsh, nsh * shb, shb))
        out["config3"] = c3
        for p in paths:
            os.unlink(p)
        del gen
        torch.cuda.empty_cache()

        # ---------------- config 5: 1000 x 128 MB blobs (pull-side verify) ---------------------------------------------
        nb, bb = args.compat5_blobs, int(args.compat5_blob_mb * 1e6)
        mine = [i for i in range(nb) if i % world == rank]
        distinct = min(16, max(1, len(mine)))
        gen = torch.empty(max(bb, 8) // 8 * 8 + 8, dtype=torch.uint8, device=dev)
        base_files = []
        for k in range(distinct):
            p = os.path.join(d, f"distinct-{k}.bin")
            eng.dev_gen_fill(0, gen.data_ptr(), ((rank * 16 + k) * bb) // 8 * 8, (bb + 7) // 8 * 8, SEED + 5, torch.cuda.current_stream().cuda_stream)
            with open(p, "wb") as f:
                f.truncate(bb)
            write_device_range_to_file(torch, gen, bb, p, 0)
            base_files.append(p)
        paths = []
        for j, i in enumerate(mine):
            p = os.path.join(d, f"blob-{i:04d}")
            os.link(base_files[j % distinct], p)
            paths.append(p)
        want = eng.sha256_files(base_files)[0] if base_files else []
        want_list = [want[j % distinct] for j in range(len(mine))]
        barrier()
        ok = eng.verify_files(paths, want_list) if paths else []          # warm-up + correctness
        if not all(ok):
            raise SystemExit("compat config 5: verify_files reported a mismatch on unmodified blobs")
        barrier()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            ok = eng.verify_files(paths, want_list) if paths else []
        dt = max_over_ranks((time.perf_counter() - t0) / reps)
        c5 = {"workload": f"{nb} x {bb/1e6:g} MB blobs, pull-side verify (pull.go:115-123), files on tmpfs; to bound tmpfs use "
                          f"the paths of a rank are hard links onto {distinct} distinct files -- every byte of every path is "
                          "still read, copied to the GPU and hashed",
              "gpu": {"value": nb * bb / dt / GB, "unit": "GB/s", "ms": dt * 1e3, "files_per_rank": len(mine),
                      "api": "mxd_verify_files (one coalesced batch per rank)"}}
        # the same 1000 paths verified by their chunked identity (tree-keyed blobs, `modelx.digest` annotation): a file is a
        # whole tree of independent leaves, so this is PCIe/host bound instead of chain-latency bound, and it scales with GPUs
        want_roots = eng.tree_digest_files(base_files)[0] if base_files else []
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            roots, _sz, st = eng.tree_digest_files(paths) if paths else ([], [], [])
        dtt = max_over_ranks((time.perf_counter() - t0) / reps)
        if any(st) or any(r != want_roots[j % distinct] for j, r in enumerate(roots)):
            raise SystemExit("compat config 5: tree-keyed verify mismatch")
        c5["gpu_tree_identity"] = {"value": nb * bb / dtt / GB, "unit": "GB/s", "ms": dtt * 1e3,
                                   "api": "mxd_tree_digest_files (all files of a rank in one pipelined pass; what mxc_pull_check runs for "
                                          "tree-keyed descriptors)"}
        if rank == 0 and paths:
            sample = paths[:24]
            tcpu, res = cpu_ref3(orc, sample)
            for (dg, _sz), w in zip(res, want_list[:len(sample)]):
                if dg != w:
                    raise SystemExit("compat config 5: GPU digest differs from the reference path on the same file")
            c5["cpu_ref_3"] = {"value": len(sample) * bb / tcpu / GB, "unit": "GB/s", "cores": 3,
                               "sample": f"{len(sample)} of the same paths, Client.digest on 3 threads; digests compared with the GPU's"}
            c5["pays_off"] = bool(modelx_b200.batch_pays_off(nb, nb * bb, bb))
        out["config5"] = c5
    finally:
        shutil.rmtree(d, ignore_errors=True)
    return out


def main():
    args = parse_args()
    import __graft_entry__ as g
    if args.impl == "reference":
        if int(os.environ.get("LOCAL_RANK", "0")) == 0:
            g.build_oracle()                      # the reference arm never builds or loads libmodelxdigest.so
        run_reference(args)
        return
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        g.build()
    run_b200(args)


if __name__ == "__main__":
    main()
