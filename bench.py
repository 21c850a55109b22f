#!/usr/bin/env python
"""bench.py — Flash Checkpoint hot path on B200.

A "step" = one memory checkpoint of this rank's shard: the Llama-3-8B bf16
state_dict (291 tensors, 16,060,522,496 bytes), resident in HBM, serialised
into the node's POSIX shared-memory segment in the reference's byte layout.

  value  whole-job checkpoint GB/s through the raw C-ABI (fc_save_async +
         fc_save_wait): gather kernel + PCIe drain, device-timed, inputs in HBM.
  e2e    the same metric through the reference-facing API
         DdpCheckpointer.save_checkpoint(step, sd, storage_type=MEMORY) +
         wait_memory_save(): shard lock RPC, readiness collective, meta publish
         (2 pickled SharedDict.set), gather kernel, D2H drain into the HOST
         shm segment, lock release.  d2h_bytes_per_step = payload; the inputs of
         this path are device-resident by definition (the model), so h2d is the
         descriptor table only (first step).
  stall_ms  what the training loop loses per checkpoint (the other half of
         BASELINE.json's metric): measured with a synthetic matmul step.
  roofline  the gather (pack) kernel against the MEASURED copy bandwidth.
  cpu_baseline / --impl reference: the reference's memory save (per-tensor
         blocking device->pageable-shm copy_) on the same box and state_dict —
         the reference's own SharedMemoryHandler from oracle/_ref/pyref (kind
         "reference"), else the restatement oracle/ref_port.py (kind "port").

Launch: python bench.py [--gpus N --steps K --warmup W] ; for N>1 under
torch.distributed.run, one rank per GPU, every rank saves its own 16 GB shard
(weak scaling, no data-path collective).

--dump-outputs DIR: rank 0 writes what its timed legs left in their segments after the
last timed step — raw_segment.npy (leg 1) and checkpoint_segment.npy (leg 2; the
reference arm writes its own segment under that name) — so that two builds can be
compared output for output on the same seeded inputs.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "checkpoint_GBps"
UNIT = "GB/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=float(os.getenv("BENCH_SCALE", "1.0")),
                    help="shrink dim 0 of every 2-D tensor (debug only; 1.0 = BASELINE config)")
    ap.add_argument("--no-stall", action="store_true", help="skip the stall measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of each segment the "
                         "timed path filled in its last step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_WORDS = 4 << 20  # 16-bit words sampled per dumped segment: 16 MB of float32 each


def dump_segment(out_dir: str, name: str, buf) -> None:
    """Writes the 16-bit words of `buf` (bf16 payload) widened bit-exactly to float32 as
    out_dir/name.npy: all of them for a small segment, else DUMP_WORDS at positions drawn
    from a fixed seed, so that two builds of the same workload dump the same positions."""
    import numpy as np

    words = np.frombuffer(buf, dtype=np.uint16, count=len(buf) // 2)
    if words.size > DUMP_WORDS:
        pos = np.sort(np.random.default_rng(20240601).integers(0, words.size, DUMP_WORDS))
        words = words[pos]
    out = (words.astype(np.uint32) << 16).view(np.float32)
    del words
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), out)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.getenv("RANK", "0"))
    local = int(os.getenv("LOCAL_RANK", "0"))
    world = int(os.getenv("WORLD_SIZE", "1"))
    return rank, local, world


def max_over_ranks(x: float, world: int, device) -> float:
    if world == 1:
        return x
    import torch
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x: float, world: int, device) -> float:
    if world == 1:
        return x
    import torch
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def barrier_sync(world):
    import torch
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (of fallback)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "pack_kernel_ncu.json")
    try:
        return json.load(open(p)).get("dram_bytes_per_launch")
    except Exception:
        return None


# ---------------------------------------------------------------- reference arm --



def reference_saver(handler_rank: int, sample):
    """The reference's own SharedMemoryHandler (byte code under oracle/_ref/pyref, built by
    oracle/build_ref.py) when it is there, imports and gets through one save of `sample`;
    otherwise the restatement oracle/ref_port.py.  Returns (saver, kind, why_not_reference)."""
    why = None
    try:
        from oracle import ref_real

        saver = ref_real.RealRefSaver(handler_rank)
        try:
            saver.save(sample)
            return saver, "reference", None
        except Exception:
            try:
                saver.close()
            except Exception:
                pass
            raise
    except Exception as e:  # noqa: BLE001
        why = f"{type(e).__name__}: {e}"[:300]
    from oracle.ref_port import RefPortSaver

    saver = RefPortSaver(f"fc_bench_ref_{os.getpid()}_{handler_rank}")
    saver.save(sample)
    return saver, "port", why


def reference_views(saver, kind):
    """Tensors aliasing the segment the reference arm wrote (ckpt_saver.py:144-161)."""
    return saver.views() if kind == "reference" else shm_layout_read(saver)


REFERENCE_HOW = {
    "reference": "the reference's own SharedMemoryHandler.save_state_dict (ckpt_saver.py:303-333, "
                 "byte code compiled from the reference by oracle/build_ref.py)",
    "port": "oracle/ref_port.py restating ckpt_saver.py:198-231,303-333",
}


def run_reference(args):
    """Times the reference's memory save on this box — the reference's own
    SharedMemoryHandler when oracle/_ref/pyref holds its byte code, else the restatement
    oracle/ref_port.py: EVERY rank runs it on its own GPU and its own shard at the same
    time (as the reference does: one blocking per-tensor copy loop per saving rank), the
    job's aggregate is reported from the slowest rank's clock."""
    rank, local, world = dist_env()
    import torch
    import torch.distributed as dist

    from dlrover_b200 import shapes

    if world > 1:
        dist.init_process_group("nccl")
    os.environ.setdefault("TORCHELASTIC_RUN_ID", f"fcbenchref{os.getppid()}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sd = {"model_states": shapes.build_state_dict(
        shapes.scale_shapes(shapes.llama3_8b_shapes(), args.scale), torch.bfloat16, dev)}
    S = shapes.payload_bytes(sd)
    saver, kind, why_port = reference_saver(200 + local, sd)  # first save: creates the segment
    # one kind for the whole job: the reference itself only if every rank runs it
    if world > 1 and sum_over_ranks(1.0 if kind == "reference" else 0.0, world, dev) != world \
            and kind == "reference":
        saver.close()
        from oracle.ref_port import RefPortSaver

        saver, kind, why_port = RefPortSaver(f"fc_bench_ref_{os.getpid()}"), "port", \
            "another rank fell back to the port"
        saver.save(sd)
    clocks = ClockSampler(local)
    try:
        for _ in range(max(args.warmup, 1)):
            saver.save(sd)
        barrier_sync(world)
        clocks.start()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            saver.save(sd)
        torch.cuda.synchronize()
        dt_mine = time.perf_counter() - t0
        barrier_sync(world)
        dt = max_over_ranks(dt_mine, world, dev)
        if args.dump_outputs and rank == 0:
            dump_segment(args.dump_outputs, "checkpoint_segment",
                         saver.buf if kind == "reference" else saver.segment.buf)
        # restore the reference's way: CPU views on the (pageable) segment, one
        # H2D copy_ per tensor (ckpt_saver.py:144-161 + model.load_state_dict)
        views = reference_views(saver, kind)
        barrier_sync(world)
        r0 = time.perf_counter()
        with torch.no_grad():
            for k, t in sd["model_states"].items():
                t.copy_(views["model_states"][k])
        torch.cuda.synchronize()
        restore_s = max_over_ranks(time.perf_counter() - r0, world, dev)
        del views
    finally:
        clk = clocks.stop()
        saver.close()
    gbs = S * world * args.steps / dt / 1e9
    if rank == 0:
        line = {
            "impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": world,
            "ranks_run": world,
            "note": f"the reference's memory-save path ({REFERENCE_HOW[kind]}) run on ALL ranks "
                    "at once, each on its own GPU and shard; value = bytes of all ranks / slowest "
                    "rank's wall time",
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": workload_config(S, world, args.scale),
            "stall_ms": {"blocking": dt / args.steps * 1e3,
                         "note": "the reference blocks the training thread for the whole copy"},
            "restore": {"reference_ms": restore_s * 1e3,
                        "reference_GBps": S * world / restore_s / 1e9,
                        "how": "frombuffer views on the pageable segment + per-tensor copy_ to "
                               "cuda, all ranks at once"},
            "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": world, "kind": kind,
                             "host_cores": os.cpu_count(), "fell_back_to_port_because": why_port,
                             "sample": f"{args.steps} full saves of the {S / 1e9:.2f} GB state_dict "
                                       f"on each of {world} rank(s): per-tensor blocking copy_ into "
                                       "a pageable /dev/shm segment, one host thread per rank "
                                       f"({REFERENCE_HOW[kind]})"},
            "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "clocks": clk,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def shm_layout_read(saver):
    """Tensors aliasing the reference-port segment (ckpt_saver.py:144-161)."""
    import torch

    from oracle.shm_layout import OracleTensorMeta, traverse

    def visit(m):
        if isinstance(m, OracleTensorMeta):
            if m.numel == 0:
                return torch.tensor([], dtype=m.dtype)
            return torch.frombuffer(saver.segment.buf, dtype=m.dtype, offset=m.offset,
                                    count=m.numel).reshape(m.shape)
        return m

    return traverse(saver.meta, visit)


def workload_config(S, world, scale):
    return {
        "workload": "Llama-3-8B bf16 state_dict (HF LlamaForCausalLM names/shapes, 291 tensors), "
                    "save every step to shared memory; BASELINE.json configs[1]"
                    + ("" if scale == 1.0 else f" [SCALED x{scale}: not the BASELINE config]"),
        "payload_bytes_per_rank": S, "ranks": world,
        "sharding": "every rank saves its own full-size shard to its own segment "
                    "(DdpCheckpointer local_shard_num=world)",
        "l2": "inputs (16 GB) and arena (16 GB) are far larger than the 126 MB L2; no flush needed",
    }


# --------------------------------------------------------------------- our arm --


def new_agent_namespace(tag: str):
    """Every leg gets its own IPC namespace (socket dir, segment names) and therefore its
    own saver daemon, forked by local rank 0 when the leg's engine is created."""
    from dlrover_b200.flash_checkpoint.engine import CheckpointEngine

    os.environ["TORCHELASTIC_RUN_ID"] = f"fcbench{os.getppid()}{tag}"
    CheckpointEngine.saver_proc = None
    return f"/tmp/fc_bench_{os.environ['TORCHELASTIC_RUN_ID']}"


def drop_segment(engine):
    """The saver daemon unlinks the segments when this process ends; do not rely on it
    alone — the driver runs several bench processes back to back on one box."""
    import torch.distributed as dist

    if dist.is_initialized():
        dist.barrier()
    shm = engine._shm_handler.shared_memory
    if shm is not None and engine._local_rank == engine.local_shard_id:
        try:
            shm.unlink()
        except (FileNotFoundError, OSError):
            pass
    engine.close()


def run_ours(args):
    rank, local, world = dist_env()
    os.environ.setdefault("TORCHELASTIC_RUN_ID", f"fcbench{os.getppid()}")
    os.environ.setdefault("DLROVER_LOG_LEVEL", "WARNING")
    # NCCL_DEBUG is left as the launcher set it (its log lines share stdout with the one
    # JSON line; rank 0 prints that line between two barriers, when NCCL is quiet)
    import torch
    import torch.distributed as dist

    if world > 1:
        os.environ.setdefault("LOCAL_WORLD_SIZE", str(world))
        dist.init_process_group("nccl")
    # create the checkpointer (forks the saver daemon on local rank 0) BEFORE
    # this process touches CUDA
    from dlrover_b200 import _native as native
    from dlrover_b200 import shapes
    from dlrover_b200.flash_checkpoint.api import DdpCheckpointer, StorageType

    ckpt_dir = f"/tmp/fc_bench_{os.getenv('TORCHELASTIC_RUN_ID')}"
    ckpt = DdpCheckpointer(ckpt_dir, local_shard_num=world, global_shard_num=world)

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sd = shapes.build_state_dict(shapes.scale_shapes(shapes.llama3_8b_shapes(), args.scale),
                                 torch.bfloat16, dev)
    S = shapes.payload_bytes(sd)
    stream = torch.cuda.current_stream()
    ctx = native.get_context(local)
    if os.getenv("BENCH_ONLY") == "coop" and world > 1:
        # development shortcut (not the driver's contract): only the cooperative leg
        ckpt.engine.close()
        coop = measure_cooperative(args, sd, S, world, dev)
        if rank == 0:
            print(json.dumps({"metric": METRIC, "n_gpus": world, "only": "ddp_cooperative",
                              "ddp_cooperative": coop}), flush=True)
        dist.barrier()
        dist.destroy_process_group()
        return 0

    # ---- leg 1: raw C-ABI (value, roofline) ------------------------------------------
    import ctypes
    import mmap

    import _posixshmem

    seg_name = f"/fc_bench_raw_{os.getpid()}"
    fd = _posixshmem.shm_open(seg_name, os.O_CREAT | os.O_EXCL | os.O_RDWR, mode=0o600)
    os.ftruncate(fd, S)
    seg = mmap.mmap(fd, S)
    addr = ctypes.addressof(ctypes.c_char.from_buffer(seg))
    t0 = time.perf_counter()
    ctx.host_register(addr, S, prefault_threads=min(16, os.cpu_count() or 1))
    register_s = time.perf_counter() - t0
    leaves = list(sd.values())
    offs, o = [], 0
    for t in leaves:
        offs.append(o)
        o += t.numel() * t.element_size()
    ctx.arena_reserve(S)
    plan = ctx.plan([t.data_ptr() for t in leaves], offs,
                    [t.numel() * t.element_size() for t in leaves])

    def raw_step():
        tk = plan.save_async(addr, stream)
        ctx.save_wait(tk)
        return ctx.save_timings(tk)

    for _ in range(max(args.warmup, 3)):
        raw_step()
    clocks = ClockSampler(local)
    barrier_sync(world)
    clocks.start()
    k0, m0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    packs, drains = [], []
    for _ in range(args.steps):
        p, d, _tot = raw_step()
        packs.append(p)
        drains.append(d)
    ev1.record(stream)
    barrier_sync(world)
    raw_ms = ev0.elapsed_time(ev1)
    k1, m1 = ctx.launch_count()
    clk = clocks.stop()
    raw_ms = max_over_ranks(raw_ms, world, dev)
    value = S * world * args.steps / raw_ms / 1e6
    pack_ms = sum(packs) / len(packs)
    drain_ms = sum(drains) / len(drains)
    peak, peak_src = measured_peak()
    achieved = 2 * S / pack_ms / 1e6

    # image check: the segment equals the device bytes (first/last tensors + checksum)
    import numpy as np

    img = np.frombuffer(seg, dtype=np.uint8)
    for t, off in ((leaves[0], offs[0]), (leaves[-1], offs[-1]), (leaves[5], offs[5])):
        n = min(t.numel() * t.element_size(), 1 << 20)
        want = t.view(-1).view(torch.uint8)[:n].cpu().numpy()
        assert np.array_equal(img[off:off + n], want), "segment image mismatch"
    del img
    if args.dump_outputs and rank == 0:
        dump_segment(args.dump_outputs, "raw_segment", seg)
    plan.destroy()
    ctx.host_unregister(addr)
    seg.close()
    os.close(fd)
    _posixshmem.shm_unlink(seg_name)

    # ---- leg 2: through the Checkpointer API (e2e) -------------------------------------
    def api_step(step):
        ckpt.save_checkpoint(step, sd, storage_type=StorageType.MEMORY)
        ckpt.wait_memory_save()

    t0 = time.perf_counter()
    api_step(1)  # creates the segment (first touch through bounce slots), builds the plan
    first_save_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    pinned = ckpt.engine.wait_segment_pinned(120)  # background pin: steady state from here
    background_pin_s = time.perf_counter() - t0
    for i in range(max(args.warmup, 3)):
        api_step(2 + i)
    barrier_sync(world)
    k2, _ = ctx.launch_count()
    t0 = time.perf_counter()
    for i in range(args.steps):
        api_step(100 + i)
    barrier_sync(world)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    k3, _ = ctx.launch_count()
    if args.dump_outputs and rank == 0:
        dump_segment(args.dump_outputs, "checkpoint_segment",
                     ckpt.engine._shm_handler.shared_memory.buf)
    e2e_ms = max_over_ranks(e2e_ms, world, dev)
    e2e = S * world * args.steps / e2e_ms / 1e6
    api_timings = ckpt.engine.last_save_timings()

    # ---- leg 2b: restore from memory (metric iv of SURVEY §8d) ---------------------------
    restore = measure_restore(ckpt, sd, S, world)

    # ---- leg 3: exposed stall with a synthetic training step ----------------------------
    stall = None
    if not args.no_stall:
        stall = measure_stall(ckpt, sd, S, dev, world)

    # ---- leg 3b: restore in a FRESH process (a restarted trainer), N=1 only ------------------
    fresh = None
    if world == 1:
        fresh = auxiliary(measure_fresh_restore, ckpt, sd, S, ckpt_dir)

    # ---- leg 4: cpu_baseline (rank 0, N=1 only) ------------------------------------------
    cpu_base = None
    if world == 1:
        cpu_base = auxiliary(measure_cpu_baseline, sd, S)

    drop_segment(ckpt.engine)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": raw_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": workload_config(S, world, args.scale),
        "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": S,
                "api": "DdpCheckpointer.save_checkpoint(MEMORY)+wait_memory_save",
                "first_save_s": first_save_s,
                "background_pin_s": background_pin_s, "pinned": bool(pinned),
                "note": "inputs of this path are the live device-resident parameters; "
                        "the host buffer is the shm segment the drain fills"},
        "stall_ms": stall,
        "restore": restore,
        "restore_fresh_process": fresh,
        "ddp_cooperative": None,
        "fsdp": None,
        "roofline": {"bound": "hbm", "kernel": "fc_copy_tma<0> (gather/pack)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": ncu_traffic(),
                     "traffic_source": "static: profiles/pack_kernel_ncu.json (one ncu --set "
                                       "full capture of this kernel on this workload, "
                                       "dram__bytes_read.sum + dram__bytes_write.sum)",
                     "algorithmic_bytes_per_launch": 2 * S, "avg_launch_ms": pack_ms,
                     "peak_source": peak_src},
        "drain": {"avg_ms": drain_ms, "GBps": S / drain_ms / 1e6, "bound": "PCIe Gen5 x16"},
        "cpu_baseline": cpu_base,
        "gpu_launches": (k1 - k0) + (k3 - k2),
        "dma_copies": m1 - m0,
        "segment_pin_s": register_s,
        "api_last_timings_ms": api_timings,
        "clocks": clk,
    }
    if world == 1:
        print(json.dumps(line), flush=True)
        return 0

    # The contract's numbers are complete here.  The two legs below (N>1) run under a
    # deadline: whatever happens in them, rank 0 prints the line and every rank exits 0.
    guard = AuxDeadline(rank, world, line)
    guard.start()
    # ---- leg 5: the SAME replicated state saved cooperatively ------------------------------
    guard.run("ddp_cooperative", measure_cooperative, args, sd, S, world, dev)
    # ---- leg 6: BASELINE configs[2] — FSDP full-shard, every rank its local shard -----------
    if not os.getenv("BENCH_NO_FSDP"):
        del sd
        torch.cuda.empty_cache()
        guard.run("fsdp", measure_fsdp, args, world, rank, local, dev)
    guard.park_if_failed()
    dist.barrier()
    guard.finish()  # prints on rank 0
    dist.barrier()  # nothing else writes to stdout while rank 0 prints
    dist.destroy_process_group()
    return 0


class AuxDeadline:
    """Keeps the legs beyond the contract's line (cooperative, FSDP) from taking the
    headline numbers down with them.  They are full of collectives: a rank that fails
    leaves the others waiting inside NCCL, where no exception can reach them.  So

      * a failing rank records the error, drops a flag file and runs no further leg;
      * a watcher thread on every rank ends the process (exit code 0) when the deadline
        (BENCH_AUX_DEADLINE_S, default 300 s) passes or GRACE seconds after any rank's
        flag appeared — rank 0 prints the line first, with what it has and an "error"
        record for what is missing;
      * when everything went well, finish() prints the line once."""

    GRACE = 15.0

    def __init__(self, rank: int, world: int, line: dict):
        self.rank, self.world, self.line = rank, world, line
        self.t_start = time.time()
        self.deadline = self.t_start + float(os.getenv("BENCH_AUX_DEADLINE_S", "300"))
        self.flags = (f"/tmp/fc_bench_flags_{os.getenv('TORCHELASTIC_RUN_ID', '')}_"
                      f"{os.getenv('MASTER_PORT', '')}_{os.getppid()}")
        self.lock = threading.Lock()
        self.printed = False
        self.failed = False
        self.running = None

    def start(self):
        os.makedirs(self.flags, exist_ok=True)
        threading.Thread(target=self._watch, daemon=True).start()

    def run(self, key, leg, *a):
        if self.failed:
            return
        self.running = key
        rec = auxiliary(leg, *a)
        with self.lock:
            if not self.printed:
                self.line[key] = rec
        self.running = None
        if isinstance(rec, dict) and "error" in rec:
            self.failed = True
            try:
                open(os.path.join(self.flags, str(self.rank)), "w").close()
            except OSError:
                pass

    def park_if_failed(self):
        """A rank whose leg failed must not enter another collective: it waits here for
        the watcher (which sees its flag) to end the process."""
        while self.failed:
            time.sleep(0.2)

    def _emit(self, why):
        with self.lock:
            if self.printed:
                return
            self.printed = True
            if self.rank == 0:
                for key in ("ddp_cooperative", "fsdp"):
                    if self.line.get(key) is None and (why or key == self.running):
                        self.line[key] = {"error": why or "not run"}
                print(json.dumps(self.line), flush=True)

    def _flagged(self):
        out = []
        try:
            for name in sorted(os.listdir(self.flags)):
                try:  # a leftover of an older run with the same ids does not count
                    if os.path.getmtime(os.path.join(self.flags, name)) >= self.t_start - 1.0:
                        out.append(name)
                except OSError:
                    pass
        except OSError:
            pass
        return out

    def _watch(self):
        # runs until the process ends: also after finish(), so that a rank waiting in the
        # last barrier for one that the deadline took away does not sit out NCCL's timeout
        first_flag = None
        while True:
            time.sleep(0.25)
            now = time.time()
            why = None
            if now > self.deadline:
                why = f"deadline: leg {self.running} still running after BENCH_AUX_DEADLINE_S"
            else:
                flagged = self._flagged()
                if flagged:
                    first_flag = first_flag or now
                    if len(flagged) == self.world or now - first_flag > self.GRACE:
                        why = f"leg abandoned: rank(s) {','.join(flagged)} failed in it"
            if why:
                self._emit(why)
                sys.stdout.flush()
                os._exit(0)

    def finish(self):
        self._emit(None)
        if self.rank == 0:
            import shutil

            shutil.rmtree(self.flags, ignore_errors=True)


def auxiliary(leg, *a):
    """The legs beyond the contract's line (cooperative, FSDP, fresh-process restore) must
    not take the headline numbers down with them: a failure becomes an "error" record."""
    try:
        return leg(*a)
    except Exception as e:  # noqa: BLE001
        import traceback

        return {"error": f"{type(e).__name__}: {e}", "where": traceback.format_exc()[-600:]}


def measure_cooperative(args, sd, S, world, dev):
    """The path configs[1] shards by at N>1: the state is REPLICATED (DDP), the reference
    lets local rank 0 alone write it (one PCIe link, full_ckpt_engine.py:76-89); here all
    local ranks drain 1/N of the same image into the same segment."""
    import torch

    from dlrover_b200.flash_checkpoint.api import DdpCheckpointer, StorageType

    ckpt = DdpCheckpointer(new_agent_namespace("c"))  # local_shard_num=1: one image per node
    assert ckpt.engine._cooperative(), "cooperative saves are off"

    def step(i):
        t0 = time.perf_counter()
        ckpt.save_checkpoint(i, sd, storage_type=StorageType.MEMORY)
        call = time.perf_counter() - t0
        ckpt.wait_memory_save()
        return call

    t0 = time.perf_counter()
    step(1)
    first = time.perf_counter() - t0
    ckpt.engine.wait_segment_pinned(120)
    for i in range(max(args.warmup, 3)):
        step(2 + i)
    barrier_sync(world)
    t0 = time.perf_counter()
    calls = [step(100 + i) for i in range(args.steps)]
    barrier_sync(world)
    dt = max_over_ranks(time.perf_counter() - t0, world, dev)
    timings = ckpt.engine.last_save_timings() or (None, None, None)
    # every rank checks ITS slice of the one image against its own replica
    import numpy as np

    shm = ckpt.engine._shm_handler.shared_memory
    img = np.frombuffer(shm.buf, dtype=np.uint8)
    lo, hi = __import__("dlrover_b200.shm_handler", fromlist=["CoopContext"]).CoopContext(
        None, ckpt.engine._local_rank, world, 0).window(S)
    ok, off = True, 0
    for t in sd.values():
        n = t.numel() * t.element_size()
        a, b = max(off, lo), min(off + n, hi)
        if b > a:
            m = min(b - a, 1 << 18)
            flat = t.view(-1).view(torch.uint8)
            ok = ok and np.array_equal(img[a:a + m], flat[a - off:a - off + m].cpu().numpy())
        off += n
    ok = bool(sum_over_ranks(0.0 if ok else 1.0, world, dev) == 0)
    del img
    # cooperative restore: every rank needs the WHOLE image back; each reads 1/N of it from
    # host memory and the slices are all-gathered between the arenas over NVLink
    keys = list(sd)
    probe = [sd[k].clone() for k in (keys[0], keys[len(keys) // 2], keys[-1])]
    restores = []
    for _ in range(3):
        for t in sd.values():
            t.zero_()
        barrier_sync(world)
        t0 = time.perf_counter()
        step_back = ckpt.load_checkpoint_into(sd)
        torch.cuda.synchronize()
        restores.append(max_over_ranks(time.perf_counter() - t0, world, dev))
    restored_ok = step_back > 0 and all(
        torch.equal(sd[k], p) for k, p in zip((keys[0], keys[len(keys) // 2], keys[-1]), probe))
    restored_ok = bool(sum_over_ranks(0.0 if restored_ok else 1.0, world, dev) == 0)
    restore_stats = dict(ckpt.engine._shm_handler.last_restore_stats)
    out = {"value": S * args.steps / dt / 1e9, "unit": UNIT,
           "restore": {"ms": min(restores) * 1e3, "first_ms": restores[0] * 1e3,
                       "GBps_per_rank": S / min(restores) / 1e9,
                       "what": "load_checkpoint_into on every rank at once: each rank gets the "
                               "whole image back (slowest rank's wall time)",
                       "bit_exact_spot_check": restored_ok, "device_times": restore_stats},
           "what": f"ONE {S / 1e9:.2f} GB image (replicated state) per node, {world} ranks each "
                   "gather + drain 1/N of it into the same segment; value = image bytes / wall "
                   "time of save_checkpoint(MEMORY)+wait_memory_save (slowest rank)",
           "ms_per_save": dt / args.steps * 1e3, "host_call_ms": sum(calls) / len(calls) * 1e3,
           "first_save_s": first, "slice_bytes": hi - lo,
           "pack_ms_slice": timings[0], "drain_ms_slice": timings[1],
           "single_link_reference_policy_ms": S / 55.5e9 * 1e3,
           "image_matches_replicas": ok}
    drop_segment(ckpt.engine)
    return out


def measure_fsdp(args, world, rank, local, dev):
    """BASELINE configs[2]: Llama-3-8B FSDP full-shard — every rank saves ITS shard (bf16
    weights + fp32 AdamW moments, rows sharded 1/N) through FsdpCheckpointEngine /
    torch.distributed.checkpoint, with fresh tensors at every save (fc_plan_update)."""
    import torch
    import torch.distributed as dist
    from torch.distributed.device_mesh import init_device_mesh

    from dlrover_b200 import shapes
    from dlrover_b200.common.constants import CheckpointConstant
    from dlrover_b200.common.storage import PosixDiskStorage
    from dlrover_b200.flash_checkpoint.fsdp_engine import FsdpCheckpointEngine

    mesh = init_device_mesh("cuda", (world,))
    factory = shapes.ShardedStateFactory(
        shapes.scale_shapes(shapes.llama3_8b_shapes(), args.scale), world, rank, dev, mesh)
    states = [factory.build(0), factory.build(1)]
    ckpt_dir = new_agent_namespace("f")
    engine = FsdpCheckpointEngine(ckpt_dir, PosixDiskStorage())
    name = CheckpointConstant.MODEL_STATES_NAME
    S_rank = factory.local_bytes

    def step(i):
        # ranks leave the previous drain at slightly different times (36-40 GB/s per link):
        # line them up like a training step's collectives would, so that `call` is the work
        # of the call and not the wait for the slowest rank inside its readiness all-reduce
        dist.barrier()
        t0 = time.perf_counter()
        ok = engine.save_to_memory(i, states[i & 1], {name: os.path.join(ckpt_dir, str(i))})
        call = time.perf_counter() - t0
        engine.wait_memory_save()
        assert ok
        return call

    t0 = time.perf_counter()
    step(1)
    first = time.perf_counter() - t0
    engine.wait_segment_pinned(120)
    for i in range(max(args.warmup, 3)):
        step(2 + i)
    barrier_sync(world)
    t0 = time.perf_counter()
    calls = [step(100 + i) for i in range(args.steps)]
    barrier_sync(world)
    dt = max_over_ranks(time.perf_counter() - t0, world, dev)
    timings = engine.last_save_timings() or (None, None, None)
    total = sum_over_ranks(float(S_rank), world, dev)
    # spot check: the items of this rank's segment are the local shards of the last save
    import numpy as np

    last = states[(100 + args.steps - 1) & 1]
    meta = engine._shm_handler.metadata.get()["dcp_metadata"]
    img = np.frombuffer(engine._shm_handler.shared_memory.buf, dtype=np.uint8)
    locals_ = factory.local_tensors(last)
    ok, checked = True, 0
    for index, info in meta.storage_data.items():
        if info.relative_path != f"__{rank}_0.distcp" or index.fqn not in locals_ or not info.length:
            continue
        t = locals_[index.fqn]
        m = min(info.length, 1 << 16)
        ok = ok and np.array_equal(img[info.offset:info.offset + m],
                                   t.reshape(-1).view(torch.uint8)[:m].cpu().numpy())
        checked += 1
    del img
    ok = bool(sum_over_ranks(0.0 if (ok and checked) else 1.0, world, dev) == 0)
    out = {"value": total * args.steps / dt / 1e9, "unit": UNIT,
           "what": "Llama-3-8B FSDP full-shard (BASELINE configs[2]): per rank 1/N of the bf16 "
                   "weights and of the fp32 AdamW moments as DTensor shards, saved through "
                   "FsdpCheckpointEngine.save_to_memory (torch DCP planning + SharedMemoryWriter: "
                   "one plan re-target, one gather kernel, one drain per rank), fresh tensors at "
                   "every save; value = bytes of all ranks / wall time (slowest rank)",
           "payload_bytes_per_rank": S_rank, "payload_bytes_total": total,
           "ms_per_save": dt / args.steps * 1e3,
           "host_call_ms": sum(calls) / len(calls) * 1e3,
           "host_call_ms_max": max(calls) * 1e3,
           "host_call_ms_slowest_rank": max_over_ranks(sum(calls) / len(calls), world, dev) * 1e3,
           "first_save_s": first,
           "pack_ms": timings[0], "drain_ms": timings[1], "items_checked": checked,
           "segment_matches_local_shards": ok}
    drop_segment(engine)
    return out


def measure_fresh_restore(ckpt, sd, S, ckpt_dir):
    """A restarted trainer: new process, attaches to the segment the dead one left in
    shared memory, restores 16 GB into live tensors.  Ours (staged bounce slots, no 16 GB
    cudaHostRegister up front) vs the reference's way (CPU views on the pageable segment +
    per-tensor copy_)."""
    import torch

    keys = list(sd)
    probe = {k: int(sd[k].view(-1).view(torch.int16)[:4096].to(torch.int64).sum().item())
             for k in (keys[0], keys[len(keys) // 2], keys[-1])}
    spec = {"probe": probe, "ckpt_dir": ckpt_dir, "scale": float(os.getenv("BENCH_SCALE", "1.0"))}
    out = {}
    for mode in ("ours", "reference_style"):
        env = dict(os.environ, FC_FRESH_SPEC=json.dumps(spec), FC_FRESH_MODE=mode)
        t0 = time.time()
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fresh_restore.py")],
                           env=env, capture_output=True, text=True, timeout=600)
        wall = time.time() - t0
        try:
            rec = json.loads(p.stdout.strip().split("\n")[-1])
        except Exception:
            rec = {"error": (p.stderr or p.stdout)[-800:]}
        rec["process_wall_s"] = wall
        out[mode] = rec
    return out


def measure_stall(ckpt, sd, S, dev, world):
    """Synthetic training loop: `inner` bf16 8192^3 matmuls per step on the
    training stream.  Compare step time without checkpoints, with an async
    memory checkpoint every `every` steps (ours), and with a blocking one."""
    import torch

    from dlrover_b200.flash_checkpoint.api import StorageType

    a = torch.randn(8192, 8192, device=dev, dtype=torch.bfloat16)
    b = torch.randn(8192, 8192, device=dev, dtype=torch.bfloat16) * 0.01
    inner, rounds = 40, 6

    grad = torch.zeros(4 << 20, device=dev) if world > 1 else None

    def train_step():
        c = a
        for _ in range(inner):
            c = torch.mm(c, b)
        if grad is not None:
            # DDP-style gradient all-reduce: keeps the ranks in lockstep like a
            # real data-parallel step does (without it they drift apart and the
            # checkpoint's readiness collective measures that drift)
            import torch.distributed as dist

            dist.all_reduce(grad)
        # like `loss.item()` in a real loop: the host does not run ahead of
        # the device by more than one step
        return float(c[0, 0].item())

    # size the checkpoint interval so a drain (S over PCIe) always fits in it
    for _ in range(3):
        train_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        train_step()
    torch.cuda.synchronize()
    step_s = (time.perf_counter() - t0) / 5
    drain_s = S / 45e9
    every = int(drain_s * 1.5 / step_s) + 2

    def loop(save_mode):
        # save_mode: None | "async" | "blocking"
        barrier_sync(world)
        t0 = time.perf_counter()
        host_in_call, saves = 0.0, 0
        for i in range(every * rounds):
            train_step()
            if save_mode and i % every == every - 1:
                before = ckpt.engine._cached_step
                h0 = time.perf_counter()
                ckpt.save_checkpoint(10_000 + i + (0 if save_mode == "async" else 100_000), sd,
                                     storage_type=StorageType.MEMORY)
                if save_mode == "blocking":
                    ckpt.wait_memory_save()
                host_in_call += time.perf_counter() - h0
                saves += int(ckpt.engine._cached_step != before)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ckpt.wait_memory_save()
        return dt, host_in_call, saves

    loop(None)
    base = min(loop(None)[0], loop(None)[0])
    asy, asy_host, n_a = loop("async")
    blk, blk_host, n_b = loop("blocking")
    timings = ckpt.engine.last_save_timings() or (None, None, None)
    return {
        "async": max((asy - base) / max(n_a, 1) * 1e3, 0.0),
        "blocking": (blk - base) / max(n_b, 1) * 1e3,
        "host_call_ms_async": asy_host / max(n_a, 1) * 1e3,
        "pack_kernel_ms": timings[0],
        "train_step_ms": base / (every * rounds) * 1e3,
        "checkpoint_every_steps": every,
        "saves_done": [n_a, n_b],
        "saves_attempted": rounds,
        "method": f"{every * rounds} synthetic steps of {inner} bf16 8192^3 matmuls + a "
                  "loss.item()-style host read per step, a memory "
                  f"checkpoint every {every} steps; stall = (loop wall time - wall time of the "
                  "same loop without checkpoints) / #checkpoints; 'async' = product default "
                  "(returns after enqueueing the gather kernel), 'blocking' = waits for the "
                  "drain inside the step like the reference",
    }


def measure_restore(ckpt, sd, S, world):
    """In-memory restore of the shard: ours = load_checkpoint_into (H2D DMA from the
    pinned segment straight into the live tensors for few large ones, arena + scatter
    kernel for many small ones); reference style =
    load_checkpoint() (CPU views on the segment) + per-tensor copy_ to the
    device, which is what model.load_state_dict does."""
    import torch

    keys = list(sd)
    probe = [sd[k].clone() for k in (keys[0], keys[7], keys[-1])]
    for t in sd.values():
        t.zero_()
    barrier_sync(world)
    t0 = time.perf_counter()
    step = ckpt.load_checkpoint_into(sd)
    torch.cuda.synchronize()
    ours = time.perf_counter() - t0
    ok = step > 0 and all(torch.equal(sd[k], p) for k, p in zip((keys[0], keys[7], keys[-1]), probe))
    out = {"ours_ms": ours * 1e3, "ours_GBps": S / ours / 1e9, "bit_exact_spot_check": bool(ok),
           "device_times": dict(ckpt.engine._shm_handler.last_restore_stats)}
    if world == 1:
        barrier_sync(world)
        t0 = time.perf_counter()
        loaded = ckpt.load_checkpoint()
        with torch.no_grad():
            for k, t in sd.items():
                t.copy_(loaded[k])
        torch.cuda.synchronize()
        ref = time.perf_counter() - t0
        del loaded
        out.update({"reference_style_ms": ref * 1e3, "reference_style_GBps": S / ref / 1e9})
    return out


def measure_cpu_baseline(sd, S):
    """Reference algorithm on this box, bounded sample: 2 full saves."""
    import torch

    wrapped = {"model_states": sd}
    saver, kind, why_port = reference_saver(150, wrapped)  # creates + faults the pageable segment
    try:
        torch.cuda.synchronize()
        n = 2
        t0 = time.perf_counter()
        for _ in range(n):
            saver.save(wrapped)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / n
    finally:
        saver.close()
    return {"value": S / dt / 1e9, "unit": UNIT, "cores": 1, "host_cores": os.cpu_count(),
            "kind": kind, "fell_back_to_port_because": why_port, "ms_per_step": dt * 1e3,
            "torch_save": measure_torch_save(sd),
            "sample": f"2 full saves of the same state_dict through {REFERENCE_HOW[kind]}: "
                      "per-tensor blocking copy_ device->pageable /dev/shm; single host thread, "
                      "as the reference"}


def measure_torch_save(sd, budget_bytes=2 << 30):
    """B0 of SURVEY §8(d): naive blocking torch.save of device tensors to /dev/shm, on a
    bounded sample (leading tensors of the state_dict up to ~2 GiB)."""
    import torch

    sample, size = {}, 0
    for k, v in sd.items():
        if size + v.numel() * v.element_size() > budget_bytes and sample:
            continue
        sample[k] = v
        size += v.numel() * v.element_size()
    path = f"/dev/shm/fc_bench_torch_save_{os.getpid()}.pt"
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        torch.save(sample, path)
        dt = time.perf_counter() - t0
    finally:
        if os.path.exists(path):
            os.remove(path)
    return {"value": size / dt / 1e9, "unit": UNIT, "bytes": size, "ms": dt * 1e3,
            "sample": f"torch.save of {len(sample)} tensors ({size / 1e9:.2f} GB) to /dev/shm"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
