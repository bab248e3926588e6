#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 collective / tensor-transport layer.

Metric (BASELINE.json): "allreduce bus GB/s vs msg size; Ray Train ResNet-50 img/s at 1/2/4/8 B200".
  value / e2e        ResNet-50 DDP synthetic-image training throughput (whole job, weak scaling),
                     gradients reduced by the fused peer-memory hook (ant_ray_b200.ddp_hook); e2e copies
                     every step's batch from pinned host memory (side stream, double-buffered) and reads
                     the step's loss back;
  allreduce_sweep    bus GB/s vs message size: ours on plain torch tensors, ours on tensors from the
                     communicator's symmetric pool (zero-copy NVLS), stock NCCL — same processes, same
                     sizes (N >= 2); two loopback ranks on the one GPU (N = 1);
  collectives        broadcast / allgather / reducescatter next to the reference's NCCL call pattern;
  p2p                2-rank B200Communicator.send/recv in the shape of the reference's compiled-graph GPU
                     microbenchmark (fp16, 100,000 bytes) + a size sweep, next to torch.distributed NCCL;
  comm_bound         the same training step at the reference harness's default batch 32, fp32 and bf16
                     gradient wire, ours next to stock NCCL DDP (where the collective is not hidden);
  parity             (N >= 2, untimed) every algorithm of the multi-GPU path checked against the NCCL
                     result of the same seeded buffers: integers bit-exact, fp32 max relative error,
                     identical bits on all ranks; hooked-DDP gradients against stock DDP;
  roofline           the dominant kernel of OUR path (the fused gradient reduction), timed live with
                     CUDA events on the stream it is launched on, back to back;
  cpu_baseline       the reference's CPU path (torch DDP over gloo, which is what Ray Train's
                     _TorchBackend selects without GPUs: train/torch/config.py:167-176) on the
                     box's host cores, bounded sample, N = 1 only.

Launch:  python bench.py --gpus 1 --steps K --warmup W
         python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
             --master-port P bench.py --gpus N --steps K --warmup W
         python bench.py --impl reference ...      (the reference's CPU path, rank 0 only)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RESNET50_PARAMS = 25_557_032
NVLINK_PEAK_MEASURED = 770.0   # GB/s per direction per GPU, peer copy (B200_PROFILING.md)
NVLINK_PEAK_NOMINAL = 900.0
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the N = 1 roofline kernel, from the committed
# `ncu --set full` capture (profiles/r02_ncu_full_local_scale_tma_details.txt: k_local_scale_tma<float, bf16_t>, 30 MiB bucket):
# 31.47 MB read; the 31.46 MB written are still dirty in the 126 MB L2 when the kernel ends (ncu: 0.00 MB)
NCU_TRAFFIC_LOCAL_SCALE_30MIB = 31_465_216 + 1_792_000   # read + write of the second of four captured launches


def log(msg):
    if int(os.environ.get("RANK", 0)) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--batch", type=int, default=int(os.environ.get("BENCH_BATCH", 256)), help="per-GPU batch")
    p.add_argument("--wire", default=os.environ.get("BENCH_WIRE", "bf16"), choices=["bf16", "fp32", "fp16"])
    p.add_argument("--no-sweep", action="store_true")
    p.add_argument("--no-nccl-ddp", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-parity", action="store_true")
    p.add_argument("--no-p2p", action="store_true")
    p.add_argument("--no-comm-bound", action="store_true")
    p.add_argument("--sweep-max-bytes", type=int, default=int(os.environ.get("BENCH_SWEEP_MAX", 1 << 30)))
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what their last step computed to DIR/<name>.npy (float32)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed regions
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None
        self.stop_evt = threading.Event()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return self
        threading.Thread(target=self._read, daemon=True).start()
        return self

    def _read(self):
        for line in self.proc.stdout:
            if self.stop_evt.is_set():
                break
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        self.stop_evt.set()
        if self.proc is not None:
            self.proc.terminate()

    def summary(self, windows):
        sm, smax, reasons = [], 0.0, set()
        for ts, line in self.samples:
            if not any(a <= ts <= b for a, b in windows):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                smax = max(smax, float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the training workload (reference harness: release/train_tests/benchmark/image_classification/
# factory.py:41 torch.randn(B,3,224,224), :372 torchvision resnet50(weights=None); runner.py:393-403)
# ------------------------------------------------------------------------------------------------
def build_model(device, channels_last=True):
    import torch
    import torchvision

    torch.manual_seed(0)
    model = torchvision.models.resnet50(weights=None)
    model = model.to(device)
    if channels_last and device.type == "cuda":
        model = model.to(memory_format=torch.channels_last)
    return model


def make_step(model, opt, use_autocast, device):
    import torch
    import torch.nn.functional as F

    def step(x, y):
        if use_autocast:
            with torch.autocast(device.type, dtype=torch.bfloat16):
                loss = F.cross_entropy(model(x), y)
        else:
            loss = F.cross_entropy(model(x), y)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    return step


def fence(dist, world):
    import torch

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(value, dist, world):
    import torch

    if world > 1:
        t = torch.tensor([value], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()
    return value


def timed_steps(step, x, y, steps, dist, world, last=None):
    """Device-resident inputs: exactly `steps` steps between two fences, CUDA events, max over ranks.
    If `last` is a list, what the final step returned is appended to it."""
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence(dist, world)
    t0 = time.time()
    e0.record()
    out = None
    for _ in range(steps):
        out = step(x, y)
    e1.record()
    fence(dist, world)
    t1 = time.time()
    if last is not None:
        last.append(out)
    return max_over_ranks(e0.elapsed_time(e1), dist, world), (t0, t1)


DUMP_PARAM_SAMPLE = 1 << 20   # 4 MB of float32; all of ResNet-50's parameters would be 102 MB


def dump_outputs(out_dir, model, loss):
    """What the training step hands back to its caller, as float32 .npy files: the loss, the batch-norm running
    statistics (every one of them) and a fixed, seeded sample of the updated parameters, whose values carry the
    gradients the fused reduction produced.  Element order is the order of model.parameters() / model.buffers()."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)

    def save(name, t):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to("cpu", torch.float32).numpy())

    save("loss", loss.reshape(1))
    save("bn_running_stats", torch.cat([b.reshape(-1).float() for b in model.buffers() if b.is_floating_point()]))
    params = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()]).cpu()
    pick = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_PARAM_SAMPLE].sort().values
    save("params_sample", params[pick])


def timed_steps_e2e(step, x_host, y_host, steps, dist, world, device):
    """End to end through the public API: every step's batch comes from pinned host memory (H2D inside the
    timed region, on a side stream, double-buffered so the copy of step i+1 overlaps step i) and every
    step's loss goes back to pinned host memory (D2H inside the timed region, asynchronous; the host reads
    the values after the final fence instead of stalling the GPU queue once per step)."""
    import torch

    copy_stream = torch.cuda.Stream(device=device)
    cur_stream = torch.cuda.current_stream(device)
    bufs = [(torch.empty_like(x_host, device=device), torch.empty_like(y_host, device=device)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.empty(steps, dtype=torch.float32).pin_memory()

    def prefetch(slot, first=False):
        with torch.cuda.stream(copy_stream):
            if not first:
                copy_stream.wait_event(consumed[slot])   # the step that read this slot has finished
            bufs[slot][0].copy_(x_host, non_blocking=True)
            bufs[slot][1].copy_(y_host, non_blocking=True)
            ready[slot].record(copy_stream)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence(dist, world)
    t0 = time.time()
    e0.record()
    prefetch(0, first=True)
    for i in range(steps):
        slot = i & 1
        cur_stream.wait_event(ready[slot])
        if i + 1 < steps:
            prefetch(slot ^ 1, first=(i == 0))
        loss = step(bufs[slot][0], bufs[slot][1])
        consumed[slot].record(cur_stream)
        loss_host[i].copy_(loss.detach().float(), non_blocking=True)
    e1.record()
    fence(dist, world)
    t1 = time.time()
    return max_over_ranks(e0.elapsed_time(e1), dist, world), (t0, t1), float(loss_host[-1])


# ------------------------------------------------------------------------------------------------
# collective timing helpers
# ------------------------------------------------------------------------------------------------
def sweep_sizes(max_bytes):
    s, out = 1024, []
    while s <= max_bytes:
        out.append(s)
        s *= 4
    return out


def time_collective(fn, bufs, iters, dist, world, rounds=2):
    """Microseconds per call: every call is bracketed by its own CUDA events (on the launching stream);
    the figure is the median over `iters` calls, best of `rounds` rounds, max over ranks.  Medians and
    a second round keep a transient on the shared host (a ~50 ms slow window was observed once per
    few sweeps, on NCCL and on our kernels alike) from landing in a single size's number."""
    import torch

    best = None
    for _ in range(rounds):
        for i in range(min(5, iters)):
            fn(bufs[i % len(bufs)])
        fence(dist, world)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for i, (e0, e1) in enumerate(evs):
            e0.record()
            fn(bufs[i % len(bufs)])
            e1.record()
        torch.cuda.synchronize()
        ts = sorted(e0.elapsed_time(e1) * 1e3 for e0, e1 in evs)
        us = max_over_ranks(ts[len(ts) // 2], dist, world)
        best = us if best is None else min(best, us)
    return best


def time_back_to_back(fn, bufs, iters, dist, world, rounds=3):
    """Microseconds per call over a back-to-back loop of `iters` launches (one event pair around the loop,
    so launch latency is hidden behind the previous kernel, as it is inside a training step), best of `rounds`."""
    import torch

    best = None
    for _ in range(rounds):
        for i in range(3):
            fn(bufs[i % len(bufs)])
        fence(dist, world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(bufs[i % len(bufs)])
        e1.record()
        torch.cuda.synchronize()
        us = max_over_ranks(e0.elapsed_time(e1) * 1e3 / iters, dist, world)
        best = us if best is None else min(best, us)
    return best


def time_torch_copy_same_size(nbytes, dist, world):
    """torch's own out-of-place copy of the same number of bytes, back to back (read nbytes + write nbytes): what a
    plain STREAM-style kernel reaches at THIS size — the driver's MEASURED_PEAKS figure is a 2 GiB copy, whose
    ramp-up and launch gap are amortised over ~650 us instead of ~10 us."""
    import torch

    n = nbytes // 4
    src = [torch.randn(n, device="cuda") for _ in range(4)]
    dst = [torch.empty(n, device="cuda") for _ in range(4)]
    us = time_back_to_back(lambda i: dst[i].copy_(src[i]), list(range(4)), 40, dist, world)
    return 2 * nbytes / (us * 1e-6) / 1e9


def time_fused_bucket(comm, dist, world, wire):
    """The fused gradient kernel alone (full grid, nothing else on the GPU) on ResNet-50's largest bucket
    (30 MiB fp32), in place, rotating over 8 buckets (240 MiB > L2).  Microseconds per launch, back to back."""
    import torch

    from ant_ray_b200 import _native as N

    n = 30 << 18
    wire_code = {"bf16": N.BFLOAT16, "fp16": N.FLOAT16, "fp32": N.FLOAT32}[wire]
    bufs = [torch.randn(n, device="cuda") for _ in range(8)]
    us = time_back_to_back(lambda b: comm.allreduce_scaled(b.data_ptr(), b.data_ptr(), n, N.FLOAT32, wire_code, 1.0 / world, N.ALGO_AUTO),
                           bufs, 40, dist, world)
    return us, n


def run_sweep_multi(comm, dist, world, max_bytes):
    """N >= 2: in-place fp32 SUM allreduce, ours (AUTO) on plain torch tensors, ours on a tensor from the
    communicator's symmetric pool (same call, zero-copy NVLS), and torch c10d NCCL on the plain tensors."""
    import torch

    from ant_ray_b200 import _native as N

    rows = []
    sym_cap = int(comm.lib.b200c_comm_symmetric_bytes(comm.handle))
    for size in sweep_sizes(max_bytes):
        n = size // 4
        nbuf = max(1, min(16, (256 << 20) // size))  # rotate buffers so small sizes are not L2-resident replays
        bufs = [torch.ones(n, dtype=torch.float32, device="cuda") for _ in range(nbuf)]
        iters = 100 if size <= (1 << 20) else (30 if size <= (64 << 20) else 8)
        ours = time_collective(lambda b: comm.allreduce(b.data_ptr(), b.data_ptr(), n, N.FLOAT32, N.SUM, N.ALGO_AUTO), bufs, iters, dist, world)
        nccl = time_collective(lambda b: dist.all_reduce(b), bufs, iters, dist, world)
        k = 2 * (world - 1) / world
        row = {"bytes": size, "b200_us": round(ours, 2), "nccl_us": round(nccl, 2),
               "b200_busbw": round(size / ours / 1e3 * k, 2), "nccl_busbw": round(size / nccl / 1e3 * k, 2)}
        if comm.multicast and size <= sym_cap and size >= (1 << 20) and size % 16 == 0:
            nsym = max(1, min(nbuf, sym_cap // size))
            sbufs = [comm.symmetric_tensor((n,), torch.float32, byte_offset=i * size) for i in range(nsym)]
            for b in sbufs:
                b.fill_(1.0)
            sym = time_collective(lambda b: comm.allreduce(b.data_ptr(), b.data_ptr(), n, N.FLOAT32, N.SUM, N.ALGO_AUTO), sbufs, iters, dist, world)
            row["b200_sym_us"], row["b200_sym_busbw"] = round(sym, 2), round(size / sym / 1e3 * k, 2)
        rows.append(row)
        del bufs
    return rows


def run_other_collectives(comm, dist, world):
    """broadcast / allgather / reducescatter next to the reference's call pattern on NCCL (allgather into a flat
    buffer + W copies, W copies + reducescatter: nccl_collective_group.py:278-296, 319-337)."""
    import torch

    from ant_ray_b200 import _native as N

    rows = []
    for size in (1 << 20, 64 << 20):
        n = size // 4
        nbuf = max(1, min(8, (256 << 20) // size))
        bufs = [torch.ones(n, device="cuda") for _ in range(nbuf)]
        iters = 50 if size <= (1 << 20) else 10
        ours = time_collective(lambda b: comm.broadcast(b.data_ptr(), n, N.FLOAT32, 0), bufs, iters, dist, world)
        ref = time_collective(lambda b: dist.broadcast(b, 0), bufs, iters, dist, world)
        rows.append({"op": "broadcast", "bytes": size, "b200_us": round(ours, 2), "nccl_us": round(ref, 2),
                     "b200_busbw": round(size / ours / 1e3, 1), "nccl_busbw": round(size / ref / 1e3, 1)})
        per = size // world // 4 * 4
        m = per // 4
        outs = [torch.empty(m, device="cuda") for _ in range(world)]
        flat = torch.empty(m * world, device="cuda")
        src = torch.ones(m, device="cuda")
        ptrs = [o.data_ptr() for o in outs]
        kf = (world - 1) / world
        ours = time_collective(lambda b: comm.allgather(src.data_ptr(), ptrs, m, N.FLOAT32), [None], iters, dist, world)

        def ref_ag(_):
            dist.all_gather_into_tensor(flat, src)
            for j in range(world):
                outs[j].copy_(flat[j * m:(j + 1) * m])

        ref = time_collective(ref_ag, [None], iters, dist, world)
        rows.append({"op": "allgather", "bytes_total": per * world, "b200_us": round(ours, 2), "nccl_ref_us": round(ref, 2),
                     "b200_busbw": round(per * world / ours / 1e3 * kf, 1), "nccl_ref_busbw": round(per * world / ref / 1e3 * kf, 1)})
        o = torch.empty(m, device="cuda")
        ours = time_collective(lambda b: comm.reducescatter(ptrs, o.data_ptr(), m, N.FLOAT32, N.SUM), [None], iters, dist, world)

        def ref_rs(_):
            for j in range(world):
                flat[j * m:(j + 1) * m].copy_(outs[j])
            dist.reduce_scatter_tensor(o, flat)

        ref = time_collective(ref_rs, [None], iters, dist, world)
        rows.append({"op": "reducescatter", "bytes_total": per * world, "b200_us": round(ours, 2), "nccl_ref_us": round(ref, 2),
                     "b200_busbw": round(per * world / ours / 1e3 * kf, 1), "nccl_ref_busbw": round(per * world / ref / 1e3 * kf, 1)})
    return rows


def run_sweep_loopback(max_bytes):
    """N = 1: two loopback ranks on the one GPU run the same kernels through local HBM."""
    import torch

    from ant_ray_b200 import _native as N
    from ant_ray_b200.loopback import LoopbackWorld

    W = 2
    world = LoopbackWorld(W, device=0, key="bench-sweep", staging_bytes=128 << 20)
    rows = []
    try:
        for size in sweep_sizes(min(max_bytes, 256 << 20)):
            n = size // 4
            bufs = [torch.ones(n, dtype=torch.float32, device="cuda") for _ in range(W)]
            iters = 100 if size <= (1 << 20) else (20 if size <= (64 << 20) else 5)

            def once():
                world.run(lambda r, c: c.allreduce(bufs[r].data_ptr(), bufs[r].data_ptr(), n, N.FLOAT32, N.SUM, N.ALGO_AUTO))

            for _ in range(3):
                once()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                once()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / iters
            rows.append({"bytes": size, "b200_us": round(us, 2), "b200_busbw": round(size / us / 1e3, 2), "loopback_ranks": W})
        world.check()
    finally:
        world.destroy()
    return rows


# ------------------------------------------------------------------------------------------------
# p2p: the reference's compiled-graph GPU microbenchmark shape
# (release/microbenchmark/experimental/compiled_graph_gpu_microbenchmark.py:71-112, 441-451)
# ------------------------------------------------------------------------------------------------
def run_p2p(dist, world, rank, device):
    """Ranks 0 (sender) and 1 (receiver).  `exec`: the reference's NcclWorker._run body — allocate, send / recv,
    torch.cuda.synchronize — per message, fp16, 100,000 bytes, ours through B200Communicator.send/recv and NCCL
    through torch.distributed.send/recv.  `sweep`: device-timed GB/s for larger messages."""
    import torch

    from ant_ray_b200.communicator import B200Communicator

    ids = [B200Communicator.generate_communicator_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    comm = B200Communicator(world, ids[0], rank, list(range(world)), torch.cuda.current_stream(), False)
    alloc = lambda shape, dtype: torch.empty(shape, dtype=dtype, device=device)  # noqa: E731
    out = {"harness": "compiled_graph_gpu_microbenchmark.py NcclWorker.do_send_recv: alloc + send/recv + cuda synchronize per message"}
    try:
        n = 100_000 // 2

        def ours():
            if rank == 0:
                comm.send(torch.ones(n, dtype=torch.float16, device=device), 1)
            elif rank == 1:
                comm.recv((n,), torch.float16, 0, alloc)
            torch.cuda.synchronize()

        def nccl():
            if rank == 0:
                dist.send(torch.ones(n, dtype=torch.float16, device=device), 1)
            elif rank == 1:
                dist.recv(torch.empty(n, dtype=torch.float16, device=device), 0)
            torch.cuda.synchronize()

        for name, fn in (("b200", ours), ("nccl", nccl)):
            for _ in range(20):
                fn()
            fence(dist, world)
            iters = 300
            t0 = time.perf_counter()
            for _ in range(iters):
                fn()
            us = (time.perf_counter() - t0) / iters * 1e6
            out[f"{name}_100kB_fp16_us_per_msg"] = round(max_over_ranks(us if rank < 2 else 0.0, dist, world), 2)
        rows = []
        for size in (1 << 20, 16 << 20, 64 << 20, 256 << 20):
            m = size // 2
            nbuf = max(1, min(4, (256 << 20) // size))
            bufs = [torch.ones(m, dtype=torch.float16, device=device) for _ in range(nbuf)]
            from ant_ray_b200.b200_group import TensorView

            def o(b):
                v = TensorView(b)
                if rank == 0:
                    comm._comm.send(v.ptr, size, 1)
                elif rank == 1:
                    comm._comm.recv(v.ptr, size, 0)

            def r(b):
                if rank == 0:
                    dist.send(b, 1)
                elif rank == 1:
                    dist.recv(b, 0)

            iters = 30 if size <= (16 << 20) else 10
            a = time_back_to_back(o, bufs, iters, dist, world, rounds=2)
            b = time_back_to_back(r, bufs, iters, dist, world, rounds=2)
            rows.append({"bytes": size, "b200_us": round(a, 2), "nccl_us": round(b, 2), "b200_gbps": round(size / a / 1e3, 1), "nccl_gbps": round(size / b / 1e3, 1)})
        out["sweep"] = rows
        comm.check()
    finally:
        comm.destroy()
    return out


# ------------------------------------------------------------------------------------------------
# parity: the multi-GPU path against the NCCL result of the same seeded buffers (untimed)
# ------------------------------------------------------------------------------------------------
def run_parity(comm, dist, world, rank, device, wire):
    """SURVEY.md 8(d) inputs: rank r draws from manual_seed(1234 + r).  For every algorithm of the path:
    int32 SUM bit-exact against ncclAllReduce of the same buffers (nccl_collective_group.py:181-188), fp32 SUM
    max |ours - nccl| / max |nccl|, and identical bits on every rank (checksum compared across ranks)."""
    import torch

    from ant_ray_b200 import _native as N

    res = {}
    g = torch.Generator().manual_seed(1234 + rank)

    def same_everywhere(t):
        s = t.view(torch.uint8).to(torch.int64).sum() if t.dtype != torch.int32 else t.to(torch.int64).sum()
        s2 = (t.view(torch.int32).to(torch.int64) * torch.arange(1, t.view(torch.int32).numel() + 1, device=t.device) % 1000003).sum()
        mine = torch.stack([s, s2])
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        return all(bool(torch.equal(v, allv[0])) for v in allv)

    def check_allreduce(name, algo, n, use_int=True, sym=False):
        entry = {}
        xf = torch.randn(n, generator=g).to(device)
        ref = xf.clone()
        dist.all_reduce(ref)
        if sym:
            cur = comm.symmetric_tensor((n,), torch.float32)
            cur.copy_(xf)
        else:
            cur = xf.clone()
        comm.allreduce(cur.data_ptr(), cur.data_ptr(), n, N.FLOAT32, N.SUM, algo)
        torch.cuda.synchronize()
        comm.check()
        entry["fp32_max_rel_err"] = float(((cur - ref).abs().max() / ref.abs().max()).item())
        entry["identical_on_all_ranks"] = same_everywhere(cur)
        if use_int:
            xi = torch.randint(-(2**15), 2**15, (n,), generator=g, dtype=torch.int32).to(device)
            refi = xi.clone()
            dist.all_reduce(refi)
            comm.allreduce(xi.data_ptr(), xi.data_ptr(), n, N.INT32, N.SUM, algo)
            torch.cuda.synchronize()
            comm.check()
            entry["int32_bit_exact"] = bool(torch.equal(xi, refi))
        entry["ok"] = entry["fp32_max_rel_err"] <= 1e-5 and entry["identical_on_all_ranks"] and entry.get("int32_bit_exact", True)
        res[name] = entry

    check_allreduce("ll", N.ALGO_LL, 4099)
    check_allreduce("oneshot", N.ALGO_ONESHOT, 100_003)
    check_allreduce("twoshot", N.ALGO_TWOSHOT, 3_000_001)
    check_allreduce("auto_1KiB", N.ALGO_AUTO, 256)
    check_allreduce("auto_64MiB", N.ALGO_AUTO, 16 << 20)
    if comm.multicast:
        check_allreduce("nvls_staged", N.ALGO_NVLS, 3_000_001, use_int=False)
        check_allreduce("nvls_rounds", N.ALGO_NVLS_PIPE, (16 << 20) + 4, use_int=False)
        check_allreduce("nvls_lanes", N.ALGO_NVLS_LANES, (24 << 20) + 12, use_int=False)
        check_allreduce("nvls_streams", N.ALGO_NVLS_STREAMS, (40 << 20) + 12, use_int=False)
        check_allreduce("auto_1GiB", N.ALGO_AUTO, 256 << 20)   # W >= 6: the multi-stream pipeline with ramped piece sizes
        check_allreduce("nvls_symmetric", N.ALGO_NVLS, 4 << 20, use_int=False, sym=True)
    # fused gradient mean, 16-bit wire: against the reference's own formulation (bf16_compress_hook:
    # buffer.to(bf16).div_(W) -> allreduce -> copy back, torch default_hooks.py)
    n = 7_500_003
    x = torch.randn(n, generator=g).to(device)
    ours = x.clone()
    wcode = {"bf16": N.BFLOAT16, "fp16": N.FLOAT16, "fp32": N.FLOAT32}[wire]
    comm.allreduce_scaled(ours.data_ptr(), ours.data_ptr(), n, N.FLOAT32, wcode, 1.0 / world, N.ALGO_AUTO)
    wdt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[wire]
    refc = x.to(wdt).div_(world)
    dist.all_reduce(refc)
    exact = x.clone()
    dist.all_reduce(exact)
    exact /= world
    torch.cuda.synchronize()
    comm.check()
    scale = exact.abs().max()
    e_ours, e_ref = float(((ours - exact).abs().max() / scale).item()), float(((refc.float() - exact).abs().max() / scale).item())
    tol = {"bf16": 2 ** -7, "fp16": 2 ** -10, "fp32": 1e-5}[wire]
    res["fused_mean_%s_wire" % wire] = {"max_rel_err_vs_fp32_mean": e_ours, "nccl_compress_hook_formulation_err": e_ref,
                                        "identical_on_all_ranks": same_everywhere(ours), "ok": e_ours <= tol and same_everywhere(ours)}
    # data movement: broadcast (small: root multicast / unicast; large: round-pipelined), allgather, reducescatter, p2p
    for name, nb in (("broadcast_1MiB", 1 << 20), ("broadcast_24MiB", 24 << 20)):
        b = torch.randint(0, 255, (nb,), generator=g, dtype=torch.uint8).to(device)
        want = b.clone()
        dist.broadcast(want, world - 1)
        comm.broadcast(b.data_ptr(), nb, N.UINT8, world - 1)
        torch.cuda.synchronize()
        comm.check()
        res[name] = {"bit_exact": bool(torch.equal(b, want)), "ok": bool(torch.equal(b, want))}
    m = 300_001
    xi = torch.randint(-1000, 1000, (m,), generator=g, dtype=torch.int32).to(device)
    outs = [torch.zeros(m, dtype=torch.int32, device=device) for _ in range(world)]
    refs = [torch.zeros(m, dtype=torch.int32, device=device) for _ in range(world)]
    dist.all_gather(refs, xi)
    comm.allgather(xi.data_ptr(), [o.data_ptr() for o in outs], m, N.INT32)
    torch.cuda.synchronize()
    ok = all(bool(torch.equal(a, b)) for a, b in zip(outs, refs))
    res["allgather"] = {"bit_exact": ok, "ok": ok}
    ins = [torch.randint(-1000, 1000, (m,), generator=g, dtype=torch.int32).to(device) for _ in range(world)]
    o, ro = torch.zeros(m, dtype=torch.int32, device=device), torch.zeros(m, dtype=torch.int32, device=device)
    dist.reduce_scatter(ro, [t.clone() for t in ins])
    comm.reducescatter([t.data_ptr() for t in ins], o.data_ptr(), m, N.INT32, N.SUM)
    torch.cuda.synchronize()
    comm.check()
    res["reducescatter"] = {"bit_exact": bool(torch.equal(o, ro)), "ok": bool(torch.equal(o, ro))}
    payload = torch.randint(0, 255, (5_000_017,), generator=torch.Generator().manual_seed(99), dtype=torch.uint8).to(device)
    got = torch.zeros_like(payload)
    if rank == 0:
        comm.send(payload.data_ptr(), payload.numel(), 1)
        if world > 2:
            comm.send_multi(payload.data_ptr(), payload.numel(), list(range(1, world)))
    else:
        if rank == 1:
            comm.recv(got.data_ptr(), got.numel(), 0)
            torch.cuda.synchronize()
            first = bool(torch.equal(got, payload))
            got.zero_()
        if world > 2:
            comm.recv_multi(got.data_ptr(), got.numel(), 0)
    torch.cuda.synchronize()
    comm.check()
    flags = torch.tensor([1 if (rank == 0 or (torch.equal(got, payload) if world > 2 else True)) else 0,
                          1 if (rank != 1 or first) else 0], device=device)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    res["send_recv"] = {"bit_exact": bool(flags[1].item()), "ok": bool(flags[1].item())}
    if world > 2:
        res["send_multi_%d_readers" % (world - 1)] = {"bit_exact": bool(flags[0].item()), "ok": bool(flags[0].item())}
    return res


def run_ddp_grad_parity(dist, world, rank, device):
    """Register the hook on a real DistributedDataParallel model (ResNet-50, bf16 autocast) and compare every
    parameter's .grad after a backward pass with what stock DDP produces from the SAME local gradients: the hook
    is wrapped so that each bucket is also reduced the stock way on a copy — torch's default reducer
    (`buffer.div_(W)`; allreduce) for the fp32 wire, bf16_compress_hook (`buffer.to(bf16).div_(W)`; allreduce;
    copy back) for the bf16 wire (torch default_hooks.py) — before the fused kernel runs on the bucket itself.
    Comparing two separate backward passes instead would mix in cuDNN's run-to-run nondeterminism."""
    import torch
    from torch.nn.parallel import DistributedDataParallel

    from ant_ray_b200 import ddp_hook

    out = {}
    gen = torch.Generator().manual_seed(4321 + rank)
    x = torch.randn(16, 3, 224, 224, generator=gen).to(device).contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, 1000, (16,), generator=gen).to(device)
    for wire in ("fp32", "bf16"):
        m = DistributedDataParallel(build_model(device), device_ids=[device], output_device=device)
        state = ddp_hook.make_grad_state(device=device.index, wire=wire, name="parity-" + wire)
        expected = {}

        def both(st, bucket, wire=wire, expected=expected):
            buf = bucket.buffer()
            if wire == "fp32":
                ref = buf.clone().div_(world)
                dist.all_reduce(ref)
            else:
                ref16 = buf.to(torch.bfloat16).div_(world)
                dist.all_reduce(ref16)
                ref = ref16.float()
            for p_, gview in zip(bucket.parameters(), bucket.gradients()):
                off = gview.storage_offset() - buf.storage_offset()
                expected[p_] = ref[off:off + gview.numel()]   # the bucket holds every gradient in the parameter's MEMORY order
            return ddp_hook.b200_allreduce_hook(st, bucket)

        m.register_comm_hook(state, both)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = torch.nn.functional.cross_entropy(m(x), y)
        loss.backward()
        torch.cuda.synchronize()
        state.comm.check()
        params = [p_ for p_ in m.parameters() if p_.grad is not None]
        def flat(t):  # dense tensors (contiguous or channels_last): the elements in memory order
            return t.as_strided((t.numel(),), (1,), t.storage_offset())

        num = max(float((flat(p_.grad) - expected[p_]).abs().max().item()) for p_ in params)
        den = max(float(expected[p_].abs().max().item()) for p_ in params)
        tol = 1e-5 if wire == "fp32" else 2 ** -6
        out["ddp_grads_%s_wire" % wire] = {"max_rel_err_vs_stock_ddp": num / den, "n_params": len(params), "n_buckets_launches": state.launches,
                                           "ok": num / den <= tol and len(params) == len(expected)}
        state.comm.destroy()
        del m
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# comm-bound rows: the reference harness's default batch (release/train_tests/benchmark/config.py:16)
# ------------------------------------------------------------------------------------------------
def run_comm_bound(args, dist, world, device, steps=30, warmup=8):
    import torch
    from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
    from torch.nn.parallel import DistributedDataParallel

    from ant_ray_b200 import train as b200_train

    B = 32
    rows = []
    g = torch.Generator().manual_seed(77)
    x = torch.randn(B, 3, 224, 224, generator=g).to(device).contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, 1000, (B,), generator=g).to(device)
    for wire in ("fp32", "bf16"):
        row = {"per_gpu_batch": B, "grad_wire": wire}
        model = b200_train.prepare_model(build_model(device), grad_wire=wire, wrap_single=True)
        state = model.b200_grad_state
        opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9)
        step = make_step(model, opt, True, device)
        for _ in range(warmup):
            step(x, y)
        # this step is bound by the host's launch rate, so the per-bucket event pair of `time_kernels` would be on the
        # critical path: throughput is timed without it, the hook's device time in a short second pass
        ms, _ = timed_steps(step, x, y, steps, dist, world)
        state.time_kernels, state.events = True, []
        ksteps = max(4, steps // 4)
        timed_steps(step, x, y, ksteps, dist, world)
        kt = state.kernel_times_ms()
        state.time_kernels = False
        row["b200_images_per_sec"] = round(world * B * steps / (ms / 1e3), 1)
        row["b200_ms_per_step"] = round(ms / steps, 3)
        row["b200_hook_ms_per_step"] = round(sum(t for t, _ in kt) / ksteps, 4)
        state.comm.destroy()
        del model, opt, step
        m2 = DistributedDataParallel(build_model(device), device_ids=[device], output_device=device)
        if wire == "bf16":
            m2.register_comm_hook(None, default_hooks.bf16_compress_hook)
        o2 = torch.optim.SGD(m2.parameters(), lr=0.01, momentum=0.9)
        s2 = make_step(m2, o2, True, device)
        for _ in range(warmup):
            s2(x, y)
        ms2, _ = timed_steps(s2, x, y, steps, dist, world)
        row["nccl_images_per_sec"] = round(world * B * steps / (ms2 / 1e3), 1)
        row["nccl_ms_per_step"] = round(ms2 / steps, 3)
        row["ratio"] = round(row["b200_images_per_sec"] / row["nccl_images_per_sec"], 4)
        del m2, o2, s2
        torch.cuda.empty_cache()
        rows.append(row)
    return rows


# ------------------------------------------------------------------------------------------------
# RLlib-shaped learner update (BASELINE config 5): KB-scale gradients, latency-bound
# ------------------------------------------------------------------------------------------------
def run_ppo_shape(dist, world, rank, device, steps=200, warmup=30):
    """RLlib's TorchLearner wraps the RLModule in DistributedDataParallel when num_learners > 1
    (rllib/core/learner/torch/torch_learner.py:533-553, `TorchDDPRLModule(module, **torch_ddp_kwargs)`), so a PPO
    learner's gradient reduction is one DDP bucket of a few hundred KB per update.  Model: RLlib's default PPO
    MLP (fcnet_hiddens [256, 256], separate value tower) on a CartPole-sized problem, minibatch 128, Adam.
    (a) DDP + our hook vs stock NCCL DDP: learner updates per second.  (b) the same gradient set reduced tensor
    by tensor through the ray.util.collective API (`collective.allreduce(tensor, group)`, the pattern of
    actor code that averages gradients by hand) vs torch.distributed.all_reduce on NCCL: microseconds per set."""
    import torch
    import torch.nn as nn
    from torch.nn.parallel import DistributedDataParallel

    from ant_ray_b200 import collective as col
    from ant_ray_b200 import ddp_hook

    def make():
        torch.manual_seed(0)

        class PPOModule(nn.Module):
            def __init__(self):
                super().__init__()
                self.pi = nn.Sequential(nn.Linear(4, 256), nn.Tanh(), nn.Linear(256, 256), nn.Tanh(), nn.Linear(256, 2))
                self.vf = nn.Sequential(nn.Linear(4, 256), nn.Tanh(), nn.Linear(256, 256), nn.Tanh(), nn.Linear(256, 1))

            def forward(self, obs):
                return self.pi(obs), self.vf(obs)

        return PPOModule().to(device)

    obs = torch.randn(128, 4, device=device)
    adv = torch.randn(128, device=device)

    def make_step(m, opt):
        def step():
            logits, v = m(obs)
            loss = -(torch.log_softmax(logits, -1)[:, 0] * adv).mean() + 0.5 * (v.squeeze(-1) - adv).pow(2).mean()
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
        return step

    out = {"model": "PPO MLP 4-256-256-{2,1}, minibatch 128, Adam", "grad_bytes": sum(p.numel() for p in make().parameters()) * 4}

    def rate(step):
        for _ in range(warmup):
            step()
        fence(dist, world)
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0, dist, world)
        return steps / dt

    m = DistributedDataParallel(make(), device_ids=[device], output_device=device)
    state = ddp_hook.register(m, wire="fp32", name="ppo")
    out["b200_hook_updates_per_s"] = round(rate(make_step(m, torch.optim.Adam(m.parameters(), lr=3e-4))), 1)
    state.comm.check()
    state.comm.destroy()
    del m
    m = DistributedDataParallel(make(), device_ids=[device], output_device=device)
    out["nccl_ddp_updates_per_s"] = round(rate(make_step(m, torch.optim.Adam(m.parameters(), lr=3e-4))), 1)
    del m
    # (b) per-tensor allreduce through the ray.util.collective surface
    grads = [torch.randn_like(p) for p in make().parameters()]
    name = "ppo-manual"
    col.init_collective_group(world, rank, backend="b200", group_name=name)

    def ours():
        for g in grads:
            col.allreduce(g, name)

    def nccl():
        for g in grads:
            dist.all_reduce(g)

    for tag, fn in (("b200_collective_api", ours), ("nccl_all_reduce", nccl)):
        us = time_back_to_back(lambda _: fn(), [None], 50, dist, world, rounds=2)
        out[tag + "_us_per_gradient_set"] = round(us, 1)
    out["tensors_per_set"] = len(grads)
    col.get_group_handle(name).check(synchronize=True)
    col.destroy_collective_group(name)
    return out


# ------------------------------------------------------------------------------------------------
# reference CPU path: torch DDP over gloo on the host cores (bounded sample)
# ------------------------------------------------------------------------------------------------
def effective_cores():
    """Host cores this container may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(quota) // int(period)))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except (OSError, ValueError):
            pass
    return n


def cpu_has_bf16():
    try:
        flags = open("/proc/cpuinfo").read()
    except OSError:
        return False
    return "avx512_bf16" in flags or "amx_bf16" in flags


def _cpu_worker(rank, world, port, batch, steps, warmup, threads, q, use_bf16, budget_s):
    import torch
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel

    torch.set_num_threads(threads)
    # under torchrun the parent's environment tells c10d to join the launcher's agent store as a client;
    # this private gloo group must bring up its own store instead
    for k in [k for k in os.environ if k.startswith("TORCHELASTIC_") or k in ("GROUP_RANK", "ROLE_RANK", "LOCAL_RANK", "RANK", "WORLD_SIZE",
                                                                                   "LOCAL_WORLD_SIZE", "ROLE_WORLD_SIZE", "GROUP_WORLD_SIZE")]:
        os.environ.pop(k, None)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    device = torch.device("cpu")
    model = DistributedDataParallel(build_model(device, channels_last=False))
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9)
    step = make_step(model, opt, use_autocast=use_bf16, device=device)
    g = torch.Generator().manual_seed(rank)
    x = torch.randn(batch, 3, 224, 224, generator=g)
    y = torch.randint(0, 1000, (batch,), generator=g)
    t_begin = time.time()
    for _ in range(warmup):
        step(x, y)
        if time.time() - t_begin > budget_s / 2:
            break
    dist.barrier()
    t0 = time.time()
    done = 0
    stop = torch.zeros(1)
    for _ in range(steps):
        step(x, y)
        done += 1
        # bounded sample: every rank stops together once the time budget is spent
        stop[0] = 1.0 if time.time() - t_begin > budget_s else 0.0
        dist.all_reduce(stop, op=dist.ReduceOp.MAX)
        if stop.item() > 0:
            break
    dt = time.time() - t0
    if rank == 0:
        q.put((dt, done))
    dist.destroy_process_group()


def cpu_reference(world, batch, steps, warmup, budget_s=60.0):
    """Reference CPU path for this workload: W processes, gloo process group, torch DDP default
    reducer, ResNet-50, bf16 autocast, synthetic images.  Returns (images/s, seconds/step, cores)."""
    import socket

    import torch.multiprocessing as mp

    cores = effective_cores()
    threads = max(1, cores // world)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    use_bf16 = cpu_has_bf16()
    procs = [ctx.Process(target=_cpu_worker, args=(r, world, port, batch, steps, warmup, threads, q, use_bf16, budget_s)) for r in range(world)]
    for p in procs:
        p.start()
    dt, done = q.get(timeout=budget_s * 4 + 120)
    for p in procs:
        p.join(timeout=60)
    return world * batch * done / dt, dt / done, threads * world, done, ("bf16 autocast" if use_bf16 else "fp32 (host CPU has no bf16 units)")


def workload_config(B, world, wire):
    """The workload both arms report (the reference arm runs a bounded sample of it: its own per-worker batch
    is what `per_gpu_batch` says on that arm's line)."""
    return {"workload": "Ray Train TorchTrainer-shaped ResNet-50 DDP step (prepare_model + gradient reduction hook), "
                        "synthetic randn(B,3,224,224), SGD momentum, bf16 autocast, fp32 grads",
            "model": "torchvision.resnet50", "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
            "grad_wire": wire, "grad_bytes_per_step": RESNET50_PARAMS * 4,
            "l2": "per-step working set (activations of the batch) is far larger than the 126 MB L2; "
                  "the sweeps rotate buffers totalling >= 256 MB"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    world = max(1, args.gpus)
    # N = 1: the b200 arm's own per-GPU batch (same config; the time budget bounds the number of steps instead).
    # N > 1: W gloo workers share the host's cores and memory, so the per-worker batch is cut to keep the whole
    # job at ~one batch of images in flight; that line's `config` says what it ran.
    default_batch = args.batch if world == 1 else max(16, args.batch // world)
    batch = int(os.environ.get("BENCH_CPU_BATCH", default_batch))
    ips, sps, cores, done, cpu_dtype = cpu_reference(world, batch, args.steps, args.warmup, budget_s=float(os.environ.get("BENCH_CPU_BUDGET_S", 150)))
    sample = f"{world} gloo worker(s) x batch {batch}, {done} steps after <= {args.warmup} warm-up, torch DDP default reducer, {cpu_dtype}"
    cfg = workload_config(batch, world, "fp32")   # the batch this arm really ran
    cfg.update({"reference_path": "torch DDP default reducer over a gloo process group on the host CPUs (what "
                                  "ray.train.torch.TorchConfig selects without GPUs, train/torch/config.py:167-176)",
                "b200_arm_per_gpu_batch": args.batch,
                "sample_note": "bounded sample of the b200 arm's workload: same model, step and metric, smaller per-worker batch so "
                               "that the CPU run ends within minutes"})
    print(json.dumps({
        "impl": "reference", "metric": "resnet50_ddp_train_images_per_sec", "value": round(ips, 2), "unit": "images/s",
        "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": round(sps * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(ips, 2), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    from ant_ray_b200 import _native as N
    from ant_ray_b200 import train as b200_train

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun for N > 1"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices (the b200 path has no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    os.environ.setdefault("B200COLL_TIMEOUT_MS", "60000")  # a benchmark should fail fast, not wait out the production default
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    torch.backends.cudnn.benchmark = True
    N.load()
    optional_errors = {}

    B = args.batch
    model = build_model(device)
    model = b200_train.prepare_model(model, grad_wire=args.wire, wrap_single=True)
    state = model.b200_grad_state
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9)
    step = make_step(model, opt, use_autocast=True, device=device)
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(B, 3, 224, 224, generator=g).contiguous(memory_format=torch.channels_last).pin_memory()
    y_host = torch.randint(0, 1000, (B,), generator=g).pin_memory()
    x = x_host.to(device, non_blocking=True)
    y = y_host.to(device, non_blocking=True)

    log(f"model ready, B={B}, world={world}; warm-up")
    sampler = ClockSampler(local).start() if rank == 0 else None
    for _ in range(max(3, args.warmup)):
        step(x, y)
    log("timing device-resident steps")
    # ---- device-resident inputs
    state.time_kernels = True
    state.events = []
    l0 = N.launch_count()
    if os.environ.get("BENCH_CUDA_PROFILER") == "1":  # ncu --profile-from-start off: capture the timed region only
        torch.cuda.profiler.start()
    last = []
    ms, win1 = timed_steps(step, x, y, args.steps, dist, world, last)
    if os.environ.get("BENCH_CUDA_PROFILER") == "1":
        torch.cuda.profiler.stop()
    launches = N.launch_count() - l0
    ktimes = state.kernel_times_ms()
    state.time_kernels = False
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last[0])
        log(f"outputs of the last timed step written to {args.dump_outputs}")
    log("timing end-to-end steps")
    # ---- end to end: inputs from pinned host memory every step, loss read back every step
    ms_e2e, win2, last_loss = timed_steps_e2e(step, x_host, y_host, args.steps, dist, world, device)
    value = world * B * args.steps / (ms / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)

    # ---- stock DDP reducer over NCCL on the same box (B-DDP baseline, BASELINE.md section 3)
    nccl_ddp = None
    log("stock NCCL DDP baseline")
    if not args.no_nccl_ddp:
        try:  # a failure of an optional section must not cost the headline line
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            from torch.nn.parallel import DistributedDataParallel

            m2 = DistributedDataParallel(build_model(device), device_ids=[device], output_device=device)
            if args.wire == "bf16":
                m2.register_comm_hook(None, default_hooks.bf16_compress_hook)
            o2 = torch.optim.SGD(m2.parameters(), lr=0.01, momentum=0.9)
            s2 = make_step(m2, o2, use_autocast=True, device=device)
            for _ in range(max(3, args.warmup)):
                s2(x, y)
            ms2, _ = timed_steps(s2, x, y, args.steps, dist, world)
            nccl_ddp = world * B * args.steps / (ms2 / 1e3)
            del m2, o2, s2
        except Exception as e:  # noqa: BLE001
            optional_errors["nccl_ddp"] = repr(e)[:300]
    multicast = bool(state.comm.multicast)
    del model, opt, step
    torch.cuda.empty_cache()

    comm_bound = ppo = None
    if world > 1 and not args.no_comm_bound:
        log("comm-bound rows (batch 32)")
        try:
            comm_bound = run_comm_bound(args, dist, world, device)
        except Exception as e:  # noqa: BLE001
            optional_errors["comm_bound"] = repr(e)[:300]
        log("RLlib-shaped learner update")
        try:
            ppo = run_ppo_shape(dist, world, rank, device)
        except Exception as e:  # noqa: BLE001
            optional_errors["rllib_ppo_shape"] = repr(e)[:300]

    # ---- collectives: parity, p2p, sweeps
    sweep = collectives = p2p = parity = None
    fused_alone = copy_same_size = None
    if world > 1:
        from ant_ray_b200.b200_group import PeerMemoryComm, make_config, next_comm_key

        sym_bytes = min(args.sweep_max_bytes, 1 << 30)
        sweep_comm = PeerMemoryComm(world, rank, next_comm_key("bench-sweep"), local, None, make_config(symmetric_bytes=sym_bytes))
        if not args.no_parity:
            log("parity block")
            try:
                parity = run_parity(sweep_comm, dist, world, rank, device, args.wire)
                parity.update(run_ddp_grad_parity(dist, world, rank, device))
                parity["all_ok"] = all(v.get("ok", False) for v in parity.values() if isinstance(v, dict))
            except Exception as e:  # noqa: BLE001
                optional_errors["parity"] = repr(e)[:400]
        if not args.no_p2p:
            log("p2p block")
            try:
                p2p = run_p2p(dist, world, rank, device)
            except Exception as e:  # noqa: BLE001
                optional_errors["p2p"] = repr(e)[:300]
        if not args.no_sweep:
            log("allreduce sweep")
            try:
                fused_alone = time_fused_bucket(sweep_comm, dist, world, args.wire)
                sweep = run_sweep_multi(sweep_comm, dist, world, args.sweep_max_bytes)
                collectives = run_other_collectives(sweep_comm, dist, world)
            except Exception as e:  # noqa: BLE001
                optional_errors["allreduce_sweep"] = repr(e)[:300]
        try:
            sweep_comm.check()
        except Exception as e:  # noqa: BLE001
            optional_errors["sweep_comm"] = repr(e)[:300]
        sweep_comm.destroy()
    elif rank == 0 and not args.no_sweep:
        log("allreduce sweep (loopback)")
        try:
            fused_alone = time_fused_bucket(state.comm, dist, world, args.wire)
            copy_same_size = time_torch_copy_same_size(30 << 20, dist, world)
            sweep = run_sweep_loopback(args.sweep_max_bytes)
        except Exception as e:  # noqa: BLE001
            optional_errors["allreduce_sweep"] = repr(e)[:300]

    if sampler is not None:
        sampler.stop()
    if rank == 0:
        # ---- roofline of the dominant kernel of our path: the fused reduction of the largest bucket
        wire_b = {"bf16": 2, "fp16": 2, "fp32": 4}[args.wire]
        by_size = {}
        for t_ms, nbytes in ktimes:
            by_size.setdefault(nbytes, []).append(t_ms)
        big = max(by_size) if by_size else 0
        t_big = statistics.mean(by_size[big]) if by_size else None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass

        def roofline_for(t_us, nelem, where):
            if world > 1:
                alg = 2 * (world - 1) / world * nelem * wire_b  # NVLink bytes in (== out) per GPU per launch
                ach = alg / (t_us * 1e-6) / 1e9
                return {"bound": "nvlink", "kernel": f"fused gradient allreduce ({args.wire} wire, fp32 accumulate, x1/W), "
                                                     f"{nelem * 4 >> 20} MiB fp32 bucket, {where}",
                        "achieved": round(ach, 1), "peak": NVLINK_PEAK_MEASURED, "peak_nominal": NVLINK_PEAK_NOMINAL, "unit": "GB/s",
                        "frac": round(ach / NVLINK_PEAK_MEASURED, 3), "traffic": None, "launch_us": round(t_us, 2),
                        "algorithmic_bytes": int(alg),
                        "peak_source": "measured peer copy per direction (B200_PROFILING.md), of measured; nominal 900"}
            alg = nelem * 8  # read fp32 + write fp32
            ach = alg / (t_us * 1e-6) / 1e9
            peak = peaks.get("hbm_gbs", 6650.0)
            return {"bound": "hbm", "kernel": f"k_local_scale_tma<float, {args.wire}>: fused gradient scale / wire rounding (world=1), {nelem * 4 >> 20} MiB fp32 bucket, {where}",
                    "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 3),
                    "traffic": NCU_TRAFFIC_LOCAL_SCALE_30MIB if nelem == (30 << 18) else None,
                    "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture "
                                    "(profiles/r02_ncu_full_local_scale_tma_details.txt); the written half is still dirty in L2 at kernel end",
                    "launch_us": round(t_us, 2), "algorithmic_bytes": int(alg),
                    "torch_copy_same_bytes_gbs": round(copy_same_size, 1) if copy_same_size else None,
                    "frac_of_torch_copy_same_bytes": round(ach / copy_same_size, 3) if copy_same_size else None,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)"}

        # `roofline`: the kernel timed alone, back to back (what the burst peak is comparable with);
        # `roofline_in_step`: the same kernel inside the training step, where it shares the GPU with the
        # backward pass on a small grid and waits for the slowest rank, so it is an upper bound on time.
        roofline_in_step = roofline_for(t_big * 1e3, big // 4, "inside the training step") if t_big else None
        roofline = roofline_for(fused_alone[0], fused_alone[1], "timed alone, back-to-back launches") if fused_alone else roofline_in_step
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cb = int(os.environ.get("BENCH_CPU_BATCH", 16))
            log("cpu baseline (bounded sample) ...")
            try:
                ips, sps, cores, done, cpu_dtype = cpu_reference(1, cb, 3, 1, budget_s=float(os.environ.get("BENCH_CPU_BUDGET_S", 45)))
                cpu_baseline = {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": "port",
                                "sample": f"1 gloo worker x batch {cb}, {done} steps after 1 warm-up (torch DDP default reducer, {cpu_dtype}, host CPU)"}
            except Exception as e:  # noqa: BLE001
                optional_errors["cpu_baseline"] = repr(e)[:300]
        hook_total = sum(t for t, _ in ktimes) / max(1, args.steps)
        out = {
            "metric": "resnet50_ddp_train_images_per_sec", "value": round(value, 1), "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(B, world, args.wire),
            "clocks": sampler.summary([win1, win2]) if sampler else None,
            "e2e": {"value": round(e2e, 1), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4 + y_host.numel() * 8,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / args.steps, 3), "last_loss": last_loss,
                    "input_path": "pinned host -> device on a side stream, double-buffered; loss -> pinned host every step, asynchronous"},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "roofline_in_step": roofline_in_step,
            "hook_ms_per_step": round(hook_total, 4),
            "cpu_baseline": cpu_baseline,
            "baselines": {"nccl_ddp_images_per_sec": round(nccl_ddp, 1) if nccl_ddp else None,
                          "nccl_version": ".".join(map(str, torch.cuda.nccl.version()))},
            "multicast": multicast,
            "comm_bound": comm_bound,
            "rllib_ppo_shape": ppo,
            "parity": parity,
            "p2p": p2p,
            "allreduce_sweep": sweep,
            "collectives": collectives,
        }
        if optional_errors:
            out["optional_section_errors"] = optional_errors
        print(json.dumps(out))
    state.comm.destroy()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
