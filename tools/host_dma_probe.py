"""Which host memory sustains N concurrent GPU->host drains?  Run under torchrun
(N = 1..8).  Every rank copies a 4 GiB HBM buffer to host memory of several kinds,
all ranks at once; prints per-rank and aggregate GB/s per kind.

  tmpfs        POSIX shm segment, NUMA-bound + prefaulted + cudaHostRegister'ed by
               fc_host_register (what the product uses)
  tmpfs_nonuma same, FC_NO_NUMA=1
  hostalloc    cudaHostAlloc (torch pin_memory)
  anon_thp     anonymous mmap + MADV_HUGEPAGE, registered the same way

The host's transparent-hugepage settings are reported as found; the probe never changes them.
"""
import json
import mmap
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("DLROVER_LOG_LEVEL", "WARNING")
import torch
import torch.distributed as dist

rank, local, world = int(os.getenv("RANK", 0)), int(os.getenv("LOCAL_RANK", 0)), int(os.getenv("WORLD_SIZE", 1))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
from dlrover_b200 import _native as native
from dlrover_b200.common.multi_process import SharedMemory

SIZE = int(os.getenv("PROBE_GIB", "4")) << 30
REPS = 3
ctx = native.get_context(local)
src = torch.empty(SIZE, dtype=torch.uint8, device=dev)
src.random_(0, 255)


def meminfo(*keys):
    out = {}
    for line in open("/proc/meminfo"):
        k, v = line.split(":")
        if k in keys:
            out[k] = int(v.split()[0]) // 1024  # MiB
    return out


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def timed_copy(dst):
    """All ranks start together; device-timed; returns GB/s of this rank."""
    piece = 256 << 20
    stream = torch.cuda.Stream()
    best = 0.0
    for _ in range(REPS):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            for o in range(0, SIZE, piece):
                dst[o:o + piece].copy_(src[o:o + piece], non_blocking=True)
            e1.record()
        e1.synchronize()
        best = max(best, SIZE / (e0.elapsed_time(e1) * 1e6))
    return best


def report(kind, gbs, extra=None):
    vals = [gbs]
    if world > 1:
        t = torch.tensor([gbs], device=dev, dtype=torch.float64)
        all_t = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(all_t, t)
        vals = [float(x.item()) for x in all_t]
    if rank == 0:
        print(json.dumps({"kind": kind, "n_gpus": world, "aggregate_GBps": round(sum(vals), 1),
                          "per_rank_GBps": [round(v, 1) for v in vals], **(extra or {})}),
              flush=True)


def run_tmpfs(kind, env=None):
    for k, v in (env or {}).items():
        os.environ[k] = v
    name = f"dmaprobe_{os.getppid()}_{rank}_{kind}"
    before = meminfo("ShmemHugePages")
    shm = SharedMemory(name=name, create=True, size=SIZE)
    try:
        t0 = time.time()
        ctx.host_register(shm.address, SIZE, prefault_threads=16)
        reg = time.time() - t0
        dst = torch.frombuffer(shm.buf, dtype=torch.uint8)
        gbs = timed_copy(dst)
        after = meminfo("ShmemHugePages")
        report(kind, gbs, {"register_s": round(reg, 2),
                           "ShmemHugePages_MiB": after.get("ShmemHugePages", 0) - before.get("ShmemHugePages", 0)})
        ok = bool(torch.equal(dst[:1 << 20].to(dev), src[:1 << 20]))
        assert ok
        del dst
        ctx.host_unregister(shm.address)
    finally:
        for k in (env or {}):
            os.environ.pop(k, None)
        shm.close()
        shm.unlink()


def run_hostalloc():
    dst = torch.empty(SIZE, dtype=torch.uint8).pin_memory()
    report("hostalloc", timed_copy(dst))
    del dst


def run_anon_thp():
    before = meminfo("AnonHugePages")
    m = mmap.mmap(-1, SIZE, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
    import ctypes

    addr = ctypes.addressof(ctypes.c_char.from_buffer(m))
    ctx.host_register(addr, SIZE, prefault_threads=16)  # advises HUGEPAGE, binds, faults, pins
    dst = torch.frombuffer(m, dtype=torch.uint8)
    gbs = timed_copy(dst)
    after = meminfo("AnonHugePages")
    report("anon_thp", gbs, {"AnonHugePages_MiB": after.get("AnonHugePages", 0) - before.get("AnonHugePages", 0)})
    del dst
    ctx.host_unregister(addr)


run_tmpfs("tmpfs")
run_tmpfs("tmpfs_nonuma", {"FC_NO_NUMA": "1"})
run_hostalloc()
run_anon_thp()

if rank == 0:
    print(json.dumps({"thp": {k: open(f"/sys/kernel/mm/transparent_hugepage/{k}").read().strip()
                              for k in ("enabled", "shmem_enabled", "defrag")},
                      "cmdline": open("/proc/cmdline").read().strip()[:400]}), flush=True)
if world > 1:
    dist.destroy_process_group()
