#!/usr/bin/env python
"""bench.py -- brotli-q5 compression throughput on B200 (BASELINE.json metric), one process per GPU.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's CPU path (C restatement in oracle/) on the host cores
  python bench.py --dump-outputs DIR ...    # also write the compressed stream of the last timed step to DIR (dump_outputs)

Workload (N = 1): BASELINE.json configs[1] -- 100 MB of enwik8-shaped synthetic text, quality 5, lgwin 22.
A step = one pass of the compression hot path over that input.  For N > 1 the stream is N x 100 MB, sharded with the
reference's compress_multi rule (one shard per rank, left window halo from the previous shard, byte-aligned seams);
per-GPU work is fixed => weak scaling.  `value` is measured with the input already resident in HBM; `e2e` goes through
the C ABI with pinned host buffers (H2D of the input and D2H of the compressed bytes inside the timed region) and, for
N > 1, includes the final concatenation: every rank's compressed bytes travel device-to-device over NCCL (exactly n bytes each,
no padding, no re-upload) to rank 0, which reads the whole stream back to host memory.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD_BYTES = 100_000_000
QUALITY, LGWIN = 5, 22
# one workload string for both arms (the driver compares them): BASELINE.json configs[1]
WORKLOAD = "enwik8-shaped synthetic text 100000000 bytes per GPU, quality=5, lgwin=22 (BASELINE configs[1])"
ALG_BYTES_PER_POS_MATCH = 9  # DESIGN.md: 1 B input + 4 B sorted position read + 4 B best[] write per position
CHUNK_BYTES = 24 << 20       # one k_match launch per chunk (csrc/bro_parse.cuh BRO_CHUNK_BYTES)
# dram__bytes_read.sum + dram__bytes_write.sum of one k_match launch (24 MiB chunk + 4 MiB halo) from the ncu --set full
# capture summarised in profiles/ (None until a capture of the current kernel exists)
NCU_MATCH_DRAM_BYTES_PER_LAUNCH = 774_424_320 + 669_327_104
NCU_MATCH_SOURCE = "profiles/r02x_ncu_q5.txt (ncu --set full, one k_match_shallow<16> launch: 29.4 M sorted entries, 25.2 M payload positions)"
DUMP_MAX_BYTES = 8 << 20  # stream bytes --dump-outputs writes over all ranks: 32 MiB as float32, within its 64 MB budget


def dump_outputs(out_dir, comp, rank=0, world=1):
    """--dump-outputs: what a caller of the timed path receives -- the compressed stream -- as float32 byte values
    (`compressed.npy`) and its length (`compressed_size.npy`, float64); with world > 1 every rank writes its own shard's
    stream under a `rank<r>_` prefix.  Each rank keeps at most DUMP_MAX_BYTES // world bytes, so the whole dump stays within
    DUMP_MAX_BYTES; a longer stream is represented by its bytes at that many positions drawn with a fixed seed, in stream
    order.  The positions depend on the stream length only, so two builds that produce the same stream write the same arrays."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    prefix = "rank%d_" % rank if world > 1 else ""
    limit = DUMP_MAX_BYTES // world
    b = comp.cpu().numpy()
    np.save(os.path.join(out_dir, prefix + "compressed_size.npy"), np.array([b.size], dtype=np.float64))
    if b.size > limit:
        b = b[np.sort(np.random.default_rng(0).choice(b.size, limit, replace=False))]
    np.save(os.path.join(out_dir, prefix + "compressed.npy"), b.astype(np.float32))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_port_throughput(data, cores):
    """Times the oracle's restatement of the reference path (oracle/brotli_ref.c) on `cores` host processes; each
    process compresses an equal slice (compress_multi's split, no shared state).  Returns MB/s of input."""
    import multiprocessing as mp
    n = len(data)
    slices = [(i * n // cores, (i + 1) * n // cores) for i in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(data,)) as pool:
        pool.map(_cpu_work, [(0, min(65536, n))] * cores)  # warm up: library load, tables
        t = time.perf_counter()
        sizes = pool.map(_cpu_work, slices)
        dt = time.perf_counter() - t
    return n / 1e6 / dt, sum(sizes)


_CPU = {}


def _cpu_init(data):
    from oracle.harness import Oracle
    _CPU["o"] = Oracle()
    _CPU["d"] = data


def _cpu_work(ab):
    a, b = ab
    c, _ = _CPU["o"].compress(_CPU["d"][a:b], QUALITY, LGWIN, size_hint=len(_CPU["d"]))
    return len(c)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (C restatement; the Rust crate cannot be
    built in this image) with all host threads, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from tools import datagen
    cores = min(os.cpu_count() or 1, 64)
    sample_bytes = min(WORKLOAD_BYTES, 6_000_000 * cores)
    data = datagen.enwik_like(sample_bytes)
    vals = []
    for i in range(args.warmup + args.steps):
        mbps, _ = cpu_port_throughput(data, cores)
        if i >= args.warmup:
            vals.append(mbps)
    best = len(vals) / sum(1.0 / v for v in vals)  # mean over the timed steps (total bytes / total time), like the GPU arm
    line = {
        "impl": "reference", "metric": "brotli-q5 compression throughput (input MB/s), lgwin=22", "value": round(best, 2),
        "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(sample_bytes / 1e6 / best * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_bytes": sample_bytes,
                   "note": "each step compresses a bounded sample of the workload, split over the host processes like compress_multi"},
        "cpu_baseline": {"value": round(best, 2), "unit": "MB/s", "cores": cores, "kind": "port",
                         "sample": "%d bytes of the workload split over %d processes (oracle/brotli_ref.c)" % (sample_bytes, cores)},
        "e2e": {"value": round(best, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--bytes", type=int, default=WORKLOAD_BYTES)
    ap.add_argument("--quality", type=int, default=QUALITY)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    # "text5" = BASELINE configs[1] (the metric's configuration, the default); "json9" = BASELINE configs[3]: JSON logs, quality 9,
    # 512 MiB per GPU (4 GiB over 8 GPUs), the compress_multi split across ranks
    ap.add_argument("--config", default="text5", choices=["text5", "json9"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the compressed stream of the last timed step to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the device path; --impl reference has no timed output to dump")
    if args.config == "json9":
        if args.bytes == WORKLOAD_BYTES:
            args.bytes = 512 << 20
        if args.quality == QUALITY:
            args.quality = 9
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import rust_brotli_b200 as rb
    from rust_brotli_b200 import sharding
    from tools import datagen
    from oracle.harness import sys_decompress

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    NB = args.bytes
    window = 1 << LGWIN

    # ---- synthetic stream: rank r owns shard r of a world x NB byte stream ----
    if args.config == "json9":
        block = datagen.json_logs(min(NB, 64_000_000), seed=4 + rank)
        shard = (block * (NB // len(block) + 1))[:NB]
    else:
        shard = datagen.enwik_like(NB, seed=8 + rank)
    halo = b""
    if world > 1:  # the window halo is the tail of the previous shard (compress_multi gives shard i the prefix as dictionary)
        tail = torch.frombuffer(bytearray(shard[-window:]), dtype=torch.uint8).cuda()
        recv = torch.empty(window, dtype=torch.uint8, device="cuda")
        ops = []
        if rank + 1 < world:
            ops.append(dist.P2POp(dist.isend, tail, rank + 1))
        if rank > 0:
            ops.append(dist.P2POp(dist.irecv, recv, rank - 1))
        if ops:
            for r in dist.batch_isend_irecv(ops):
                r.wait()
        if rank > 0:
            halo = bytes(recv.cpu().numpy())
    local = halo + shard
    first, last, align = sharding.shard_flags(rank, world)
    rstart = len(halo)

    enc = rb.DeviceEncoder(local_rank)
    L = rb.lib()
    h = enc._h
    cap = L.b200_max_compressed_size(NB) + 4096

    # resident buffers for `value`, pinned host buffers for `e2e`
    d_in = torch.frombuffer(bytearray(local), dtype=torch.uint8).cuda()
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    h_in = torch.frombuffer(bytearray(local), dtype=torch.uint8).pin_memory()
    h_out = torch.empty(cap, dtype=torch.uint8).pin_memory()
    osz = ctypes.c_size_t(0)

    def step_resident():
        ok = L.b200_encoder_compress_range(h, args.quality, LGWIN, NB, ctypes.c_void_p(d_in.data_ptr()), len(local), rstart, NB,
                                           int(first), int(last), int(align), ctypes.c_void_p(d_out.data_ptr()), cap,
                                           ctypes.byref(osz), 1)
        if not ok:
            raise RuntimeError("device compression failed")
        return osz.value

    # e2e: host input through the C ABI (H2D inside), compressed bytes stay on the device for the concatenation step; the whole
    # stream is then read back to host memory by rank 0.  Shard sizes are deterministic (same input every step): they are
    # exchanged once, outside the timed region.
    d_e2e_out = torch.empty(cap, dtype=torch.uint8, device="cuda")

    def compress_host_to_device(h_src):
        ok = L.b200_encoder_compress_range(h, args.quality, LGWIN, NB, ctypes.c_void_p(h_src.data_ptr()), len(local), rstart, NB,
                                           int(first), int(last), int(align), ctypes.c_void_p(d_e2e_out.data_ptr()), cap,
                                           ctypes.byref(osz), 2)
        if not ok:
            raise RuntimeError("e2e compression failed")
        return osz.value

    n_mine = compress_host_to_device(h_in)
    sizes = [n_mine]
    if world > 1:
        sz = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(sz, torch.tensor([n_mine], dtype=torch.int64, device="cuda"))
        sizes = [int(x.item()) for x in sz]
    total_out = sum(sizes)
    offs = [sum(sizes[:r]) for r in range(world)]
    d_cat = torch.empty(total_out + 16, dtype=torch.uint8, device="cuda") if rank == 0 else None   # the concatenated stream
    h_cat = torch.empty(total_out + 16, dtype=torch.uint8).pin_memory() if rank == 0 else None

    def step_e2e(h_src=None):
        n = compress_host_to_device(h_in if h_src is None else h_src)
        if world > 1:  # final concatenation: exactly n bytes per shard, device to device over NVLink
            if rank == 0:
                d_cat[:n].copy_(d_e2e_out[:n], non_blocking=True)
                ops = [dist.P2POp(dist.irecv, d_cat[offs[r]:offs[r] + sizes[r]], r) for r in range(1, world)]
            else:
                ops = [dist.P2POp(dist.isend, d_e2e_out[:n], 0)]
            for req in dist.batch_isend_irecv(ops):
                req.wait()
            if rank == 0:
                h_cat[:total_out].copy_(d_cat[:total_out], non_blocking=True)
        else:
            h_cat[:n].copy_(d_e2e_out[:n], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return n

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness once, outside the timed region ----
    n_out = step_resident()
    comp = bytes(d_out[:n_out].cpu().numpy())
    if world == 1:
        assert sys_decompress(comp, NB) == shard, "round trip failed"
    # the concatenated stream of all ranks (what step_e2e leaves on rank 0) must decode to the concatenated shards
    import hashlib
    step_e2e()
    my_sha = torch.frombuffer(bytearray(hashlib.sha256(shard).digest()), dtype=torch.uint8).cuda()
    shas = [torch.zeros(32, dtype=torch.uint8, device="cuda") for _ in range(world)]
    if world > 1:
        dist.all_gather(shas, my_sha)
    else:
        shas = [my_sha]
    roundtrip_ok = None
    if rank == 0:
        whole = sys_decompress(bytes(h_cat[:total_out].numpy()), NB * world)
        roundtrip_ok = len(whole) == NB * world and all(
            hashlib.sha256(whole[r * NB:(r + 1) * NB]).digest() == bytes(shas[r].cpu().numpy()) for r in range(world))
        assert roundtrip_ok, "concatenated stream of %d shards does not decode to the input" % world
    # ratio delta vs the reference restatement (outside the timed region): every rank compresses its own shard with the oracle
    # (for ranks > 0 without the window halo, which only makes the reference larger by a few bytes per shard)
    ref_bytes = None
    if not args.no_cpu_baseline:
        from oracle.harness import Oracle, sys_compress
        if args.config == "json9":  # bounded: the reference size of the first 64 MB, scaled to the shard (the shard repeats that block)
            ref_local = int(len(Oracle().compress(shard[:64_000_000], args.quality, LGWIN)[0]) * (NB / min(NB, 64_000_000)))
        elif args.quality <= 9:
            ref_local = len(Oracle().compress(shard, args.quality, LGWIN, size_hint=NB)[0])
        else:  # the restatement covers q4..q9; above that the stated size reference is libbrotlienc (tests/golden/make_golden.py)
            ref_local = len(sys_compress(shard, args.quality, LGWIN))
        rt = torch.tensor([float(ref_local)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(rt, op=dist.ReduceOp.SUM)
        ref_bytes = int(rt.item())

    sampler = ClockSampler(local_rank)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    # ---- value: HBM-resident.  Every call blocks until its last kernel and copy are done, so the CUDA events recorded
    # around the loop bracket exactly the device work of the K steps. ----
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler.start()
    launches = 0
    ev[0].record()
    for _ in range(args.steps):
        n_last = step_resident()
        launches += enc.timings()[1]
    ev[1].record()
    barrier()
    wall = ev[0].elapsed_time(ev[1]) * 1e-3
    clocks = sampler.stop()
    if args.dump_outputs:  # before the loops below reuse d_out
        dump_outputs(args.dump_outputs, d_out[:n_last], rank, world)
    # ---- e2e: host buffers through the C ABI ----
    for _ in range(2):
        step_e2e()
    barrier()
    ev[2].record()
    for _ in range(args.steps):
        n_e2e = step_e2e()
    ev[3].record()
    barrier()
    wall_e2e = ev[2].elapsed_time(ev[3]) * 1e-3
    # the same with pageable (not pinned) host input, as a drop-in client of the C ABI would pass it
    h_pageable = torch.frombuffer(bytearray(local), dtype=torch.uint8)
    step_e2e(h_pageable)
    barrier()
    ev_p = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev_p[0].record()
    for _ in range(args.steps):
        step_e2e(h_pageable)
    ev_p[1].record()
    barrier()
    wall_pageable = ev_p[0].elapsed_time(ev_p[1]) * 1e-3
    # ---- per-stage device times for the roofline: same workload, chunks serialised on one lane so that the CUDA events
    # around each kernel (recorded on the stream it is launched on) time that kernel alone ----
    enc.set_option(rb._native.OPT_TIMING, 1)
    enc.set_option(rb._native.OPT_LANES, 1)
    stage_acc = {}
    step_resident()
    for _ in range(args.steps):
        step_resident()
        for k, v in enc.timings()[0].items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
    barrier()

    t = torch.tensor([wall, wall_e2e, wall_pageable], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_out)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    wall, wall_e2e, wall_pageable = float(t[0]), float(t[1]), float(t[2])
    total_in = NB * world
    value = total_in * args.steps / wall / 1e6
    e2e = total_in * args.steps / wall_e2e / 1e6

    if rank == 0:
        peak, peak_src = load_peaks()
        match_ms = stage_acc.get("match", 0.0) / args.steps
        stage_ms = {k: round(v / args.steps, 3) for k, v in stage_acc.items()}
        achieved = (ALG_BYTES_PER_POS_MATCH * NB) / (match_ms * 1e-3) / 1e9 if match_ms > 0 else None
        cpu = None
        if not args.no_cpu_baseline and world == 1:  # the CPU baseline is timed at N = 1 only
            sample = shard[:16_000_000]
            mbps, _ = cpu_port_throughput(sample, 1)
            cpu = {"value": round(mbps, 2), "unit": "MB/s", "cores": 1, "kind": "port",
                   "sample": "first %d bytes of the workload, oracle/brotli_ref.c (C restatement of the reference path), 1 thread" % len(sample)}
        parse_ms = stage_acc.get("parse", 0.0) / args.steps
        dominant = "parse" if parse_ms > match_ms else "match"
        comp_total = int(float(tot[0]))
        line = {
            "metric": "brotli-q%d compression throughput (input MB/s), lgwin=22" % args.quality,
            "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(wall / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD if (NB == WORKLOAD_BYTES and args.quality == QUALITY and args.config == "text5") else
                       ("synthetic JSON logs %d bytes per GPU (a 64 MB block repeated), quality=%d, lgwin=%d (BASELINE configs[3])"
                        % (NB, args.quality, LGWIN)) if args.config == "json9" else
                       "enwik8-shaped synthetic text %d bytes per GPU, quality=%d, lgwin=%d" % (NB, args.quality, LGWIN),
                       "l2_policy": "input (100 MB) + per-position tables (>1 GB) exceed the 126 MB L2 every step",
                       "pipeline": "24 MiB chunks on 4 alternating streams (lanes); H2D staging and D2H of finished output overlap compute",
                       "sharding": "compress_multi split, one shard per GPU, 4 MiB left halo, byte-aligned seams"},
            "compressed_bytes": comp_total, "ratio": round(comp_total / total_in, 5),
            # BASELINE metric's "ratio delta %": (size_ours - size_ref) / size_ref, reference = oracle/brotli_ref.c (q <= 9; pinned to the
            # reference's KAT) or libbrotlienc (q >= 10) on the same shards
            "reference_compressed_bytes": ref_bytes,
            "ratio_delta_pct": round((comp_total - ref_bytes) * 100.0 / ref_bytes, 4) if ref_bytes else None,
            "roundtrip": {"decoder": "libbrotlidec 1.1.0", "concatenated_shards": world, "bit_exact": roundtrip_ok},
            "value_note": "device-resident input and output, no collective inside the timed region",
            "stage_ms": stage_ms,
            "dominant_stage": dominant,
            "roofline": {"bound": "hbm", "kernel": "k_match_shallow<16> (match finder, SURVEY 8d; the north-star's roofline kernel)", "achieved": round(achieved, 1) if achieved else None, "peak": peak,
                         "unit": "GB/s", "frac": round(achieved / peak, 4) if achieved else None, "traffic": NCU_MATCH_DRAM_BYTES_PER_LAUNCH,
                         "traffic_source": NCU_MATCH_SOURCE,
                         "peak_source": peak_src, "algorithmic_bytes_per_position": ALG_BYTES_PER_POS_MATCH,
                         "launch_ms": round(match_ms / max(1, -(-NB // CHUNK_BYTES)), 4),
                         "timed": "CUDA events on the launching stream, chunks serialised on one lane (K extra steps after the value loop)"},
            # the parse has the larger share of the serialised step (profiles/r02q: 31.5 % vs 27.6 %) but is latency bound (15.8 % warps
            # active, profiles/r02x_ncu_q5.txt), not a memory kernel
            "roofline_parse": {"kernel": "k_parse", "algorithmic_bytes_per_position": 6.8,
                               "achieved": round(6.8 * NB / (stage_acc.get("parse", 0.0) / args.steps * 1e-3) / 1e9, 1) if stage_acc.get("parse") else None,
                               "unit": "GB/s", "note": "1 B input + 4 B best[] + 12 B per command (0.15 commands / byte)"},
            "cpu_baseline": cpu,
            "e2e": {"value": round(e2e, 1), "unit": "MB/s", "h2d_bytes_per_step": len(local), "d2h_bytes_per_step": int(total_out if rank == 0 else 0),
                    "path": "C ABI with pinned host input (H2D inside), shard outputs device-to-device over NCCL to rank 0 (exact sizes), whole stream D2H on rank 0",
                    "pageable_input_value": round(total_in * args.steps / wall_pageable / 1e6, 1)},
            "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
