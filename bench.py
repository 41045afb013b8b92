#!/usr/bin/env python
"""bench.py — GiB/s of fused RS(12,4) encode + HighwayHash256 bitrot over 1 MiB blocks (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                    (the CPU path on the host cores; rank 0 only)

A step = one pass of the hot path over the resident synthetic stream (BASELINE config 2: 10 GiB of random object bytes per
GPU -> 10240 erasure blocks; inputs are far larger than the 126 MB L2, so no explicit flush is needed).
  value     device-resident (inputs already in HBM), CUDA events, max over ranks
  e2e       the PutObject shape through the C ABI with HOST buffers: mec_encode_sg — H2D of the object bytes, fused kernel,
            parity frames + digests back by DMA — NUMA-local pinned buffers, rank bound to its GPU's node
  e2e_frames / e2e_decode   Erasure.Encode with complete part.N images (mec_encode) and Erasure.Decode with four shards
            offline (mec_decode), same buffers
  configs   BASELINE configs 3, 4 and 5 (device-resident kernels + config 4 through mec_heal_batch), each with its own
            roofline fraction and a check against the encode outputs
  cpu_baseline / --impl reference   the C oracle's SIMD path on a persistent, pinned pthread pool over all host cores

  --dump-outputs DIR   after the timed steps, rank 0 writes a fixed sample of what the last timed step returned (parity shards
            and digests in float32, the sampled block indices in float64) as DIR/<name>.npy; the input stream is seeded, so two
            builds can be compared array for array
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K, M, BS = 12, 4, 1 << 20
S = -(-BS // K)                      # 87382
ALGO_BYTES_PER_BLOCK = BS + M * S + (K + M) * 32   # 1 398 616 (SURVEY.md §8d)
GiB = float(1 << 30)
METRIC = "fused RS(12,4) encode + HighwayHash256 bitrot, 1 MiB blocks"
# ALU-pipe warp instructions of the steady-state loop per 256-byte tile of one erasure block (LOP3 + PRMT + IADD3 + IADD3.X in the
# SASS of fused_rs_hh_kernel<GfStatic<12,4>,1,6,4,0,1>; profiles/r2_sass_loop.md says how to recount): 172 GF + 224 HighwayHash + 9 loop
ALU_WARP_INSTR_PER_TILE_BLOCK = 405
CPU_BLOCKS = int(os.environ.get("MEC_CPU_BLOCKS", "4096"))   # CPU arm: 4 GiB source per pass — larger than any last-level cache
# --dump-outputs sample, as float32: parity of 16 blocks (22.4 MB) and digests of up to 12288 blocks (25.2 MB; all of the default
# 10240), so the files stay under 64 MB whatever --blocks is
DUMP_PARITY_BLOCKS, DUMP_DIGEST_BLOCKS, DUMP_SEED = 16, 12288, 0x4D494E494F03


def workload_config(nblocks, world):
    """The same dict for both arms (the driver compares them)."""
    return {"workload": f"BASELINE config 2: RS(12,4) encode+HighwayHash256S bitrot, 1 MiB blocks, {nblocks} blocks "
                        f"({nblocks * BS / GiB:.2f} GiB stream) per GPU",
            "l2": "inputs (>=10 GiB per step) exceed the 126 MB L2; no explicit flush", "parallelism": f"sets-per-gpu x{world}"}


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        return len(self.rows)

    def summary(self, a=0, b=None):
        sm, mx, reasons = [], None, set()
        for r in self.rows[a:b]:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if not self.proc:
            return
        time.sleep(0.15)
        self.proc.terminate()


# ---------------------------------------------------------------------------------------------- CPU arm
class CpuArm:
    """The reference's two-pass CPU path (SIMD RS encode, then HighwayHash of every shard) on a persistent pool: threads are
    created and pinned once, every worker first-touches (and fills) the source blocks it will encode, timing starts when
    the workers are released.  Used by --impl reference and by the cpu_baseline leg: same pool, same buffers, same blocks."""

    def __init__(self, threads, nblocks=CPU_BLOCKS):
        import oracle_lib as o
        self.L = o.lib()   # built by build(): the benchmark compiles nothing into the tree
        self.threads, self.nblocks = threads, nblocks
        self.pool = self.L.orc_pool_new(threads)
        # untouched anonymous memory: np.empty does not touch the pages, the workers do (first touch = node-local)
        self.src = np.empty(nblocks * BS, dtype=np.uint8)
        self.parity = np.empty(nblocks * M * S, dtype=np.uint8)
        self.dig = np.empty(nblocks * (K + M) * 32, dtype=np.uint8)
        self.L.orc_pool_fill(self.pool, K, M, BS, self.src.ctypes.data, nblocks, self.parity.ctypes.data, self.dig.ctypes.data, 0x4D494E494F02)
        self.level = self.L.orc_simd_level().decode()

    def run(self, reps=1):
        sec = self.L.orc_pool_encode_hash(self.pool, K, M, BS, self.src.ctypes.data, self.nblocks, self.parity.ctypes.data, self.dig.ctypes.data, reps)
        return self.nblocks * reps * BS / GiB / sec, sec

    def describe(self, what):
        return (f"{what}; {self.nblocks} x 1 MiB blocks per pass, C oracle ({self.level}): SIMD RS encode, then HighwayHash of all 16 shards "
                f"(two passes, as the reference); {self.threads} pthreads created once, pinned over all allowed CPUs, source first-touched "
                f"by its worker; Go toolchain absent")

    def close(self):
        self.L.orc_pool_free(self.pool)


def reference_arm(args, threads):
    arm = CpuArm(threads)
    for _ in range(max(args.warmup, 1)):
        arm.run()
    secs = [arm.run()[1] for _ in range(args.steps)]
    mean = sum(secs) / len(secs)
    value = arm.nblocks * BS / GiB / mean
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * mean, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": workload_config(args.blocks, args.gpus),
        "cpu_baseline": {"value": value, "unit": "GiB/s", "cores": threads, "kind": "port",
                         "sample": arm.describe(f"each step = one pass over a {arm.nblocks} MiB sample of the workload")},
        "e2e": {"value": value, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    arm.close()


# ---------------------------------------------------------------------------------------------- helpers
def pinned(nbytes, device):
    import minio_b200 as mb
    return mb.capi.pinned_array(nbytes, device=device)


def ptr_array(arrs):
    return (C.c_void_p * len(arrs))(*[(a.ctypes.data if a is not None else None) for a in arrs])


def dump_outputs(out_dir, par, dig, nblocks):
    """What a caller of the timed encode receives, for a seeded sample of blocks: parity.npy [block, parity shard, S] (without the
    row pitch padding, which the kernel does not write), digests.npy [block, shard, 32], and the sampled block indices."""
    import torch
    rng = np.random.default_rng(DUMP_SEED)
    pb, db = (np.arange(nblocks) if n >= nblocks else np.sort(rng.choice(nblocks, n, replace=False))
              for n in (DUMP_PARITY_BLOCKS, DUMP_DIGEST_BLOCKS))
    out = {"parity": par.view(nblocks, M, -1)[torch.from_numpy(pb).to(par.device), :, :S].float().cpu().numpy(),
           "digests": dig[torch.from_numpy(db).to(dig.device)].float().cpu().numpy(),
           "parity_blocks": pb.astype(np.float64), "digest_blocks": db.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks", type=int, default=10240, help="erasure blocks per GPU per step (10240 = 10 GiB)")
    ap.add_argument("--e2e-blocks", type=int, default=2048)
    ap.add_argument("--heal-objects", type=int, default=128, help="config 4: 64 MiB objects per GPU through mec_heal_batch")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    threads = len(os.sched_getaffinity(0)) or os.cpu_count() or 1

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, threads)
        return

    import minio_b200 as mb
    L = mb.lib()
    # one rank per GPU, each bound to the CPUs (and, through first touch, the memory) of its GPU's NUMA node
    affinity0 = os.sched_getaffinity(0)
    numa_node = L.mec_bind_thread_to_device(local) if world > 1 or os.environ.get("MEC_BENCH_BIND", "1") == "1" else -1
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    nblocks = args.blocks
    nbytes = nblocks * BS
    pitch = (S + 15) // 16 * 16

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # synthetic object stream, generated on device (counter-based Philox via torch), seed per BASELINE.md §4
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x4D494E494F00 + 2 + rank)
    src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    step = 1 << 30
    for o0 in range(0, nbytes, step):
        n = min(step, nbytes - o0)
        src[o0:o0 + n] = torch.randint(0, 256, (n,), dtype=torch.uint8, device=dev, generator=gen)
    par = torch.empty((nblocks * M, pitch), dtype=torch.uint8, device=dev)
    dig = torch.empty((nblocks, K + M, 32), dtype=torch.uint8, device=dev)
    codec = mb.Codec(K, M, BS, device=local)
    stream = torch.cuda.current_stream()

    def one_step():
        codec.encode_blocks_device(src.data_ptr(), nbytes, par.data_ptr(), pitch, dig.data_ptr(), stream.cuda_stream)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    l0 = codec.launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    mark0 = sampler.mark()
    t_all0 = torch.cuda.Event(enable_timing=True); t_all1 = torch.cuda.Event(enable_timing=True)
    t_all0.record(stream)
    for a, b in evs:
        a.record(stream); one_step(); b.record(stream)
    t_all1.record(stream)
    barrier()
    mark1 = sampler.mark()
    launches = codec.launches - l0
    total_ms = max_over_ranks(t_all0.elapsed_time(t_all1))
    kern_ms = [a.elapsed_time(b) for a, b in evs]
    ms_per_step = total_ms / args.steps
    value = world * nbytes / GiB / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, par, dig, nblocks)

    # ---- input scatter over NVLink (SURVEY §8e): rank 0 owns a single-source stream and hands every rank its slice
    # with NCCL; timed separately from the kernel metric (the data path itself has no collective)
    scatter = None
    if world > 1:
        per = 1 << 30
        recv = torch.empty(per, dtype=torch.uint8, device=dev)
        chunks = [src[(i % 8) * per:(i % 8 + 1) * per] for i in range(world)] if rank == 0 else None
        for _ in range(2):
            dist.scatter(recv, chunks, src=0)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(3):
            dist.scatter(recv, chunks, src=0)
        s1.record(stream)
        barrier()
        sms = max_over_ranks(s0.elapsed_time(s1) / 3)
        scatter = {"bytes_per_rank": per, "ms": sms, "egress_GBps_rank0": (world - 1) * per / (sms / 1e3) / 1e9,
                   "note": "NCCL scatter from rank 0, timed apart from the encode kernel"}
        del recv

    # ---- the oracle as CHECKER of three blocks of the device-resident output (outside every timed region); rank 0
    verified = None
    oracle_leg = rank == 0 and not args.no_cpu
    if oracle_leg:
        import oracle_lib as o
        verified = True
        for b in (0, nblocks // 2, nblocks - 1):
            blk = src[b * BS:(b + 1) * BS].cpu().numpy()
            sh = o.encode_data(K, M, blk, fast=True)
            hp = par[b * M:(b + 1) * M, :S].cpu().numpy()
            hd = dig[b].cpu().numpy()
            for j in range(M):
                verified &= bool(np.array_equal(hp[j], sh[K + j]))
            for i in range(K + M):
                verified &= hd[i].tobytes() == o.hh256(sh[i], fast=True)

    # ---- end to end through the C ABI: NUMA-local pinned host buffers, H2D + kernel + D2H inside the timed region
    e2e = e2e_frames = e2e_decode = e2e_verify = host_link = None
    if not args.no_e2e:
        eb = min(args.e2e_blocks, nblocks)
        olen = eb * BS
        fsz = codec.bitrot_file_size(olen)
        h_src = pinned(olen, local)
        torch.from_numpy(h_src).copy_(src[:olen])
        files = [pinned(fsz, local) for _ in range(K + M)]
        h_dd = pinned(eb * K * 32, local)
        h_dst = pinned(olen, local)
        fp_all = ptr_array(files)
        fp_off = ptr_array([None if i in (0, 1, 2, 3) else files[i] for i in range(K + M)])  # GetObject with four data drives offline

        def timed(fn, reps):
            for _ in range(2):
                fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
            return max_over_ranks(time.perf_counter() - t0)

        def sg_step():
            rc = L.mec_encode_sg(codec.h, h_src.ctypes.data, olen, fp_all, h_dd.ctypes.data, K + 1)
            assert rc == olen, rc

        def frames_step():
            rc = L.mec_encode(codec.h, h_src.ctypes.data, olen, fp_all, K + 1)
            assert rc == olen, rc

        hint = C.c_int(0)

        def decode_step():
            rc = L.mec_decode(codec.h, fp_off, 0, olen, olen, h_dst.ctypes.data, C.byref(hint))
            assert rc == olen and hint.value == 0, (rc, hint.value)

        reps = args.steps
        dt = timed(sg_step, reps)
        par_bytes = M * (fsz)          # parity frames (digest + shard per block)
        e2e = {"value": world * olen * reps / GiB / dt, "unit": "GiB/s", "h2d_bytes_per_step": olen, "d2h_bytes_per_step": par_bytes + eb * K * 32,
               "call": "mec_encode_sg (Erasure.Encode, PutObject shape: parity part files + data-shard digests come back, data shards stay in the caller's buffer)",
               "sample": f"{eb} blocks ({olen / GiB:.0f} GiB object) per call per GPU, buffers from mec_alloc_pinned_on (NUMA node {numa_node}), rank bound to that node"}
        dt = timed(frames_step, max(reps // 2, 3))
        e2e_frames = {"value": world * olen * max(reps // 2, 3) / GiB / dt, "unit": "GiB/s", "h2d_bytes_per_step": olen, "d2h_bytes_per_step": (K + M) * fsz,
                      "call": "mec_encode (complete part.N images of all 16 drives written by DMA; D2H carries 1.33x the object)"}
        frames_step()
        torch.cuda.synchronize()
        if oracle_leg and verified:   # the oracle checks one whole frame of a parity drive and of a data drive, and the decode
            b = eb - 1
            sh = o.encode_data(K, M, h_src[b * BS:(b + 1) * BS], fast=True)
            for i in (K, 3):
                fr = files[i][b * (32 + S):(b + 1) * (32 + S)]
                verified &= fr[:32].tobytes() == o.hh256(sh[i], fast=True) and bool(np.array_equal(fr[32:], sh[i]))
        codec.set_option("jit", 1)
        dt = timed(decode_step, max(reps // 2, 3))
        e2e_decode = {"value": world * olen * max(reps // 2, 3) / GiB / dt, "unit": "GiB/s", "h2d_bytes_per_step": K * fsz, "d2h_bytes_per_step": olen,
                      "call": "mec_decode (Erasure.Decode, data drives 0-3 offline: 12 survivor part files in, digests verified, 4 shards rebuilt, object bytes out by DMA)"}
        if oracle_leg and verified:
            verified &= bool(np.array_equal(h_dst, h_src))
        # deep scan (bitrotVerify of every part file of the object, cmd/bitrot.go:164): hash + compare only, one byte in per byte scanned
        nfl = K + M
        fl_arr = (C.c_int64 * nfl)(*[fsz] * nfl); pl_arr = (C.c_int64 * nfl)(*[codec.shard_file_size(olen)] * nfl); res_arr = (C.c_int32 * nfl)()

        def verify_step():
            rc = L.mec_bitrot_verify_batch(codec.h, nfl, fp_all, fl_arr, pl_arr, res_arr)
            assert rc == 0 and not any(res_arr), (rc, list(res_arr))
        dt = timed(verify_step, max(reps // 2, 3))
        e2e_verify = {"value": world * nfl * fsz * max(reps // 2, 3) / GiB / dt, "unit": "GiB/s of part-file bytes scanned", "h2d_bytes_per_step": nfl * fsz, "d2h_bytes_per_step": nfl * eb,
                      "call": "mec_bitrot_verify_batch (deep scan of all 16 part files of the object; every frame's HighwayHash recomputed and compared)"}
        # what the link itself gives: pinned H2D alone, then H2D and D2H together (the pattern of the calls above)
        d_a = torch.empty(1 << 30, dtype=torch.uint8, device=dev); d_b = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
        t_src = torch.from_numpy(h_src[:1 << 30]); t_dst = torch.from_numpy(h_dst[:1 << 28])
        s2 = torch.cuda.Stream(device=dev)

        def h2d_only():
            d_a.copy_(t_src, non_blocking=True)

        def bidir():
            d_a.copy_(t_src, non_blocking=True)
            with torch.cuda.stream(s2):
                for _ in range(4):
                    t_dst.copy_(d_b, non_blocking=True)
            s2.synchronize()
        dt1 = timed(h2d_only, 5)
        dt2 = timed(bidir, 5)
        host_link = {"numa_node": numa_node, "h2d_alone_GBps": world * 5 * (1 << 30) / dt1 / 1e9, "h2d_with_d2h_GBps": world * 5 * (1 << 30) / dt2 / 1e9,
                     "d2h_with_h2d_GBps": world * 5 * (1 << 30) / dt2 / 1e9,
                     "note": "aggregate over ranks; pinned NUMA-local buffers; the e2e legs cannot exceed h2d_with_d2h (object bytes in) at 1.33x D2H per byte"}
        del d_a, d_b
        for a in files + [h_src, h_dd, h_dst]:
            L.mec_free_pinned(a.ctypes.data)

    mark2 = sampler.mark()
    # ---- BASELINE configs 3, 4, 5 (device-resident kernels; config 4 also through the host boundary)
    configs = None
    if not args.no_configs:
        del par, dig
        src = None
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_configs as bc
        bc.set_device(local)
        nb3 = min(nblocks, 8192)

        def agg(res, key="GiB_per_s_object"):
            """aggregate a per-rank device-timed result: every rank ran the same shape, the slowest rank sets the time"""
            ms = max_over_ranks(res["ms"])
            return {"value": world * res["blocks"] * res["block_size"] / GiB / (ms / 1e3), "unit": "GiB/s", "ms": ms,
                    "roofline": {"bound": "hbm", "achieved": res["algorithmic_bytes_per_block"] * res["blocks"] / (ms / 1e3) / 1e9,
                                 "frac": res["algorithmic_bytes_per_block"] * res["blocks"] / (ms / 1e3) / 1e9 / read_peaks()[0], "unit": "GB/s",
                                 "algorithmic_bytes_per_block": res["algorithmic_bytes_per_block"]},
                    "bit_exact_vs_encode": bool(res["bit_exact_vs_encode"]), "blocks_per_gpu": res["blocks"]}
        configs = {}
        r = bc.reconstruct_case("3a", 12, 4, BS, nb3, {0, 1, 2, 3}, 3, 3, quiet=True, steps=6)
        configs["3a: RS(12,4) reconstruct, data shards {0,1,2,3} erased (GetObject shape: rebuilt shards not hashed)"] = dict(agg(r), generic_kernel_GiB_per_s=r["generic_GiB_per_s"])
        r = bc.reconstruct_case("3b", 12, 4, BS, nb3, {1, 5, 12, 15}, 3, 0, quiet=True, steps=6)
        configs["3b: RS(12,4) reconstruct, shards {1,5,12,15} erased (heal shape: rebuilt shards hashed)"] = dict(agg(r), generic_kernel_GiB_per_s=r["generic_GiB_per_s"])
        r = bc.reconstruct_case("4", 16, 4, BS, nb3, {0, 7, 16, 19}, 4, 0, quiet=True, steps=6)
        configs["4-kernel: RS(16,4) heal of shards {0,7,16,19}, device-resident slice"] = dict(agg(r), generic_kernel_GiB_per_s=r["generic_GiB_per_s"])
        hb = heal_batch_leg(mb, local, args.heal_objects, barrier, max_over_ranks, world)
        configs[hb.pop("name")] = hb
        configs["small: one 1 MiB RS(12,4) PutObject / degraded GetObject per call (the shape of cmd/erasure-encode.go:76-108; latency, not throughput)"] = small_request_leg(mb, local)
        sw = bc.sha256_sweep(8, 8, [64 << 10, 256 << 10, 1 << 20, 4 << 20], 1 << 30, quiet=True)
        configs["5: RS(8,8) encode + SHA256 whole-file bitrot, block-size sweep (1 GiB per point per GPU)"] = {
            f"{r['block_size'] >> 10} KiB": {"value": world * (1 << 30) / GiB / (max_over_ranks(r["ms"]) / 1e3), "unit": "GiB/s",
                                             "roofline_frac": r["frac_of_hbm_peak"] * r["ms"] / max_over_ranks(r["ms"]),
                                             "bit_exact_vs_hashlib": bool(r["bit_exact_vs_encode"])} for r in sw}

    if rank == 0:
        sampler.stop()
    clocks = sampler.summary(mark0, mark1) if rank == 0 else None
    if rank == 0 and clocks and clocks.get("samples", 0) < 2:
        clocks = sampler.summary(mark0, mark2)   # a timed region shorter than the sampling period: take the (GPU-busy) e2e legs in as well
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = read_peaks()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    traffic_src = None
    if os.path.exists(tp):  # dram__bytes_read + dram__bytes_write of this kernel from the committed ncu capture, scaled per launch
        tj = json.load(open(tp))
        traffic = (tj["dram_bytes_read_per_block"] + tj["dram_bytes_write_per_block"]) * nblocks
        traffic_src = f"profiles/r2_traffic.json: ncu --set full capture of {tj.get('blocks')} blocks, scaled per block (not measured in this run)"
    kavg_ms = sum(kern_ms) / len(kern_ms)
    achieved = ALGO_BYTES_PER_BLOCK * nblocks / (kavg_ms / 1e3) / 1e9
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    alu_ops = ALU_WARP_INSTR_PER_TILE_BLOCK * 32 * (S / 256.0) * nblocks        # lane-ops of the steady-state loop per launch
    alu_rate = alu_ops / (kavg_ms / 1e3)
    alu_peak = 64 * 148 * sm_mhz * 1e6
    cfg = workload_config(nblocks, world)
    out = {
        "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": cfg,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_block": ALGO_BYTES_PER_BLOCK,
                     "kernel_ms": kavg_ms, "blocks_per_launch": nblocks},
        "alu_roofline": {"achieved_lane_ops_per_s": alu_rate, "peak_lane_ops_per_s": alu_peak, "frac": alu_rate / alu_peak,
                         "alu_warp_instr_per_tile_block": ALU_WARP_INSTR_PER_TILE_BLOCK,
                         "note": "the kernel is bound by the integer ALU pipe (64 lanes/clk/SM), not by HBM: this is the pipe's busy fraction from instruction counts"},
        "e2e": e2e, "e2e_frames": e2e_frames, "e2e_decode": e2e_decode, "e2e_verify": e2e_verify, "host_link": host_link,
        "gpu_launches": int(launches), "clocks": clocks, "verified_vs_oracle": verified,
    }
    if configs is not None:
        out["configs"] = configs
    if scatter:
        out["scatter"] = scatter
    if not args.no_cpu and world == 1:
        os.sched_setaffinity(0, affinity0)   # the CPU arm gets every core the process was given, not just the GPU's node
        arm = CpuArm(len(affinity0))
        arm.run()
        gib1, sec1 = arm.run()
        reps = max(1, int(10.0 / max(sec1, 1e-3)))
        gib, sec = arm.run(reps)
        split = {}
        for mode, name in ((1, "encode_only_GiB_per_s"), (2, "hash_only_GiB_per_s")):   # SURVEY §8d: the two passes apart
            arm.L.orc_pool_set_mode(mode)
            arm.run()
            split[name] = arm.run(max(1, reps // 8))[0]
        arm.L.orc_pool_set_mode(0)
        model = ""
        try:
            model = [l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
        except Exception:
            pass
        out["cpu_baseline"] = {"value": gib, "unit": "GiB/s", "cores": arm.threads, "kind": "port", "cpu_model": model, **split,
                               "sample": arm.describe(f"{reps} passes = {sec:.1f} s")}
        arm.close()
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def small_request_leg(mb, local):
    """Launches that cannot fill the GPU: kernel time of a 1-block and a 148-block encode in the latency form (ec_small.cuh) and in the
    throughput form, and the wall clock of one 1 MiB mec_encode_sg / mec_decode (four data drives offline) call from pinned buffers."""
    import torch
    k, m, bs = 12, 4, BS
    L = mb.lib()
    out = {"unit": "us"}
    for nb in (1, 148):
        src = torch.randint(0, 256, (nb * bs,), dtype=torch.uint8, device=f"cuda:{local}")
        for name, small in (("latency_form", -1), ("throughput_form", 0)):
            c = mb.Codec(k, m, bs, device=local)
            c.set_option("small_blocks", small)
            S = c.shard_size()
            pitch = (S + 15) // 16 * 16
            par = torch.zeros((nb * m * pitch,), dtype=torch.uint8, device=f"cuda:{local}")
            dig = torch.zeros((nb * (k + m) * 32,), dtype=torch.uint8, device=f"cuda:{local}")
            st = torch.cuda.current_stream()
            ts = []
            for it in range(15):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                c.encode_blocks_device(src.data_ptr(), nb * bs, par.data_ptr(), pitch, dig.data_ptr(), st.cuda_stream)
                e1.record(st)
                torch.cuda.synchronize()
                if it >= 5:
                    ts.append(e0.elapsed_time(e1) * 1e3)
            out[f"kernel_{nb}_blocks_{name}"] = round(statistics.median(ts), 1)
            c.close()
    size = bs
    c = mb.Codec(k, m, bs, device=local)
    fsz = c.bitrot_file_size(size)
    h_src = pinned(size, local)
    h_src[:] = np.random.default_rng(5).integers(0, 256, size, dtype=np.uint8)
    files = [pinned(fsz, local) for _ in range(k + m)]
    dd, dst = pinned(k * 32, local), pinned(size, local)
    assert L.mec_encode(c.h, h_src.ctypes.data, size, ptr_array(files), 0) == size
    gptrs = ptr_array([None if i < 4 else files[i] for i in range(k + m)])
    hint = C.c_int(0)
    calls = {"call_put_1MiB_mec_encode_sg": lambda: L.mec_encode_sg(c.h, h_src.ctypes.data, size, ptr_array(files), dd.ctypes.data, 0),
             "call_degraded_get_1MiB_mec_decode": lambda: L.mec_decode(c.h, gptrs, 0, size, size, dst.ctypes.data, C.byref(hint))}
    for name, fn in calls.items():
        ts = []
        for it in range(60):
            t0 = time.perf_counter()
            assert fn() == size
            if it >= 10:
                ts.append((time.perf_counter() - t0) * 1e6)
        out[name] = round(statistics.median(ts), 1)
    out["bit_exact_roundtrip"] = bool(np.array_equal(dst, h_src))
    c.close()
    for a in files + [h_src, dd, dst]:
        L.mec_free_pinned(a.ctypes.data)
    return out


def heal_batch_leg(mb, local, nobj, barrier, max_over_ranks, world):
    """BASELINE config 4 through the host boundary: `nobj` 64 MiB RS(16,4) objects per GPU with shards {0,7,16,19} stale, healed by
    mec_heal_batch over a pool of three codec handles from NUMA-local pinned part files into pinned outputs.  16 distinct
    objects are encoded and reused round-robin (the survivors still cross PCIe for every object)."""
    k, m, bs, size = 16, 4, 1 << 20, 64 << 20
    n, stale_set, distinct = k + m, (0, 7, 16, 19), 16
    enc = mb.Codec(k, m, bs, device=local)
    rng = np.random.default_rng(40 + local)
    fsz = enc.bitrot_file_size(size)
    objs, refs = [], []
    data = pinned(size, local)
    for o in range(distinct):
        data[:] = rng.integers(0, 256, size, dtype=np.uint8)
        files = [pinned(fsz, local) for _ in range(n)]
        rc = mb.lib().mec_encode(enc.h, data.ctypes.data, size, ptr_array(files), k)
        assert rc == size
        refs.append({i: files[i].copy() for i in stale_set} if o < 2 else None)
        objs.append([None if i in stale_set else files[i] for i in range(n)])
        for i in stale_set:
            mb.lib().mec_free_pinned(files[i].ctypes.data)
    enc.close()
    outs = [[pinned(fsz, local) if i in stale_set else None for i in range(n)] for _ in range(distinct)]
    stale = [i in stale_set for i in range(n)]
    npool = int(os.environ.get("MEC_HEAL_POOL", "3"))
    pool = [mb.Codec(k, m, bs, device=local) for _ in range(npool)]
    for c in pool:
        c.set_option("jit", int(os.environ.get("MEC_HEAL_JIT", "1")))
    objects = [(objs[o % distinct], stale, size) for o in range(nobj)]
    outs_all = [outs[o % distinct] for o in range(nobj)]
    mb.heal_batch(pool, objects[:6], outs_all[:6])   # warm: buffers, specialised kernel
    barrier()
    t0 = time.perf_counter()
    mb.heal_batch(pool, objects, outs_all)
    dt = max_over_ranks(time.perf_counter() - t0)
    ok = all(np.array_equal(outs[o][i], refs[o][i]) for o in range(2) for i in stale_set)
    for c in pool:
        c.close()
    for o in range(distinct):
        for a in objs[o] + outs[o]:
            if a is not None:
                mb.lib().mec_free_pinned(a.ctypes.data)
    mb.lib().mec_free_pinned(data.ctypes.data)
    return {"name": f"4-host: RS(16,4) heal batch, {nobj} objects x 64 MiB per GPU through mec_heal_batch (pool of {npool} handles, pinned NUMA-local part files)",
            "value": world * nobj * size / GiB / dt, "unit": "GiB/s of object data healed", "seconds": dt, "objects_per_gpu": nobj,
            "h2d_bytes": nobj * k * fsz, "d2h_bytes": nobj * len(stale_set) * fsz, "bit_exact_vs_encode": bool(ok)}


if __name__ == "__main__":
    main()
