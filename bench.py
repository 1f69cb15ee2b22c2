#!/usr/bin/env python3
"""bench.py -- the headline measurement of BASELINE.json on B200.

A "step" is one pass of the hot path over one batch of synthetic stripes:
  default workload  = BASELINE config C2: RS(12,4) encode + fused CRC32-IEEE of all 16 shards,
                      4 MiB blobs (shard 349,526 B, HBM pitch 349,568 B), 1024 stripes per GPU.
  --workload reconstruct = config C3 as the headline instead: same stripes, 3 random erasures per stripe.
`value`  = device-resident whole-job data throughput (k*S*stripes / t), inputs already in HBM.
`extra`  = (N=1) the other kernels of BASELINE's "encode + reconstruct" metric measured in the same run, same
           batch: plain encode, verify, C3 reconstruct (3 random erasures per stripe), single-pattern repair
           (one broken shard index for the whole batch), each with ms / data GiB/s / roofline fraction / kernel.
`checked_stripes` = stripes of the TIMED batch compared with the CPU oracle after the timed region (parity bytes,
           all 16 CRCs, reconstructed shards): first, last and seeded random ones.  A mismatch aborts the run.
`e2e`    = the same metric through the C-ABI host entry point cubeec_encode_contig on pinned HOST
           buffers (H2D of the data shards and D2H of parity + CRCs inside the timed region).
`e2e_single_call` = how access actually calls the codec (blobstore/common/ec/encoder.go:114-131): T host threads,
           each encoding ONE 4 MiB blob per cubeec_encode call from pageable memory; the engine's coalescing
           queue forms the batches.  Stripes/s, GiB/s and p50/p99 call latency.
`roofline` = algorithmic bytes ((k+m)*S per stripe for encode, (k+e)*S for reconstruct) / device time
           against the measured HBM copy bandwidth in MEASURED_PEAKS.json (and the nominal 8 TB/s).
`cpu_baseline` = the oracle's multi-threaded SIMD port (AVX2 nibble tables / GFNI as klauspost would
           select, + PCLMUL CRC32) on this box's host cores, bounded sample.

`--dump-outputs DIR` = what the last timed step handed back, for comparing two builds output for output: the parity
           shards (encode) or the regenerated shards (reconstruct) of the checked stripes and, with CRC, the CRCs of
           every shard of the batch, as DIR/<name>.npy in float32 / float64 (rank 0; 45 MB or less).  The inputs are
           seeded, so the same arguments give the same inputs on every run.

python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
python bench.py --impl reference ...                   (the reference's CPU path = oracle port; rank 0 only)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, M = 12, 4
BLOB = 4 << 20
GIB = float(1 << 30)
NOMINAL_HBM_GBS = 8000.0   # B200 HBM3e spec ceiling (BASELINE.md section 3 asks for both fractions)


def shard_size(blob, k, min_shard=2048):
    return max((blob + k - 1) // k, min_shard)   # blobstore/common/ec/buf.go:77-81


PROFILE_OF_KERNEL = {"rs_bsf_kernel<crc>": "r02_prof_bsf_crc.txt", "rs_bs_kernel<crc>": "r01_prof_r1_bs_crc.txt",
                     "rs_bs_kernel": "r02_prof_bs_nocrc.txt", "rs_tabk_kernel": "r02_prof_tabk_rec.txt",
                     "rs_jit_kernel": "r02_prof_jit_rec.txt"}


def traffic_from_profile(kernel: str, stripes: int):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel, read from the committed ncu
    --set full summary under profiles/ (taken at 1024 stripes; scaled linearly to this batch).  NOT measured in
    this run -- a profiler run is never a bench value -- hence the field name."""
    name = PROFILE_OF_KERNEL.get(kernel)
    try:
        txt = open(os.path.join(ROOT, "profiles", name)).read()
        tot = 0.0
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            for line in txt.splitlines():
                if line.startswith(key + " "):
                    val, unit = line.split()[1], line.split()[2]
                    tot += float(val) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[unit]
        return (int(tot * stripes / 1024), "profiles/" + name) if tot else (None, None)
    except Exception:
        return None, None


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region.  The sampler is started ahead of the
    region (nvidia-smi takes tens of ms to produce its first line) at a 20 ms period; samples are attributed by their
    host arrival time, and only those that arrived inside [t0, t1 + one period] count."""

    PERIOD_MS = 20

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", str(self.PERIOD_MS)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t_end = time.perf_counter() + 2.0
            while not self.rows and time.perf_counter() < t_end:   # wait for the first line
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(2.5 * self.PERIOD_MS / 1e3)
        self.proc.terminate()
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 1.5 * self.PERIOD_MS / 1e3]
        window = "timed region"
        if not inside:   # region shorter than a period: the samples on either side of it
            before = [r for (t, r) in self.rows if t < t0][-1:]
            after = [r for (t, r) in self.rows if t > t1][:1]
            inside, window = before + after, "nearest samples around a region shorter than the sampling period"
        sm, mx, reasons = [], 0, set()
        for r in inside:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------
# NUMA: pin this rank's host threads (and therefore its first-touch pinned buffers) to the GPU's node
# ---------------------------------------------------------------------------------------------------------
def pin_to_gpu_numa_node(local_rank: int):
    """SURVEY 8e "host threads pinned per device": the 8-GPU boxes are 2-socket; a rank whose staging buffers sit
    on the other socket pays the inter-socket link on every H2D/D2H.  Returns a description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank)
        pci = f"{bus.pci_domain_id:04x}:{bus.pci_bus_id:02x}:{bus.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{pci}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "single node / not reported"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"numa_node": node, "note": "node CPUs not in this process's affinity mask; left unpinned"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed), "pci": pci}
    except Exception as e:   # noqa: BLE001
        return {"numa_node": None, "note": f"unpinned ({type(e).__name__})"}


# ---------------------------------------------------------------------------------------------------------
# CPU legs (the oracle's SIMD port): cpu_baseline of the GPU arm and the whole reference arm
# ---------------------------------------------------------------------------------------------------------
class CpuLeg:
    def __init__(self, workload, stripes_sample):
        from oracle import pyoracle
        self.workload, self.sample = workload, stripes_sample
        self.S = shard_size(BLOB, K)
        self.n = K + M
        self.rs = pyoracle.RS(K, M)
        rng = np.random.default_rng(0xC0BEF5)
        self.buf = rng.integers(0, 256, (stripes_sample, self.n, self.S), dtype=np.uint8)
        self.crc = np.zeros((stripes_sample, self.n), dtype=np.uint32)
        self.present = np.ones((stripes_sample, self.n), dtype=np.uint8)
        self.cores = os.cpu_count() or 1
        if workload == "reconstruct":
            self.rs.encode_batch_simd(self.buf, self.S, self.S, self.n * self.S, stripes_sample, threads=self.cores)
            for s in range(stripes_sample):
                self.present[s, rng.choice(self.n, size=3, replace=False)] = 0
        self.REP = 4   # passes per call, so thread start-up is amortised
        self.threads = self.cores
        self._tune()

    def one(self):
        if self.workload == "encode":
            self.rs.encode_batch_simd(self.buf, self.S, self.S, self.n * self.S, self.sample, threads=self.threads,
                                      crc_out=self.crc, repeat=self.REP)
        else:
            self.rs.reconstruct_batch_simd(self.buf, self.S, self.S, self.n * self.S, self.sample, self.present,
                                           threads=self.threads, repeat=self.REP)

    def _tune(self):
        # the container may expose more CPUs than it may use: pick the thread count that is fastest
        best = None
        c = self.cores
        for th in sorted({c, max(1, c // 2), max(1, c // 4), min(c, 32), min(c, 16), min(c, 8)}):
            self.threads = th
            self.one()
            t0 = time.perf_counter()
            self.one()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, th)
        self.threads = best[1]

    def describe(self):
        return (f"oracle SIMD port ({self.rs.simd_kind()} GF kernels as klauspost v1.11.7 selects for k={K}; "
                f"PCLMUL CRC32-IEEE), one stripe per thread, {self.threads} threads")


def cpu_baseline(workload, stripes_sample, target_seconds=12.0):
    leg = CpuLeg(workload, stripes_sample)
    t0 = time.perf_counter()
    reps = 0
    while True:
        leg.one()
        reps += 1
        el = time.perf_counter() - t0
        if el >= target_seconds or reps >= 200:
            break
    reps *= leg.REP
    gibs = K * leg.S * stripes_sample * reps / el / GIB
    return {"value": round(gibs, 3), "unit": "GiB/s", "cores": leg.threads, "kind": "port",
            "sample": f"{stripes_sample} stripes x {reps} passes, {el:.1f} s, {leg.describe()}"}


def cpu_single_call(blob, seconds=3.0):
    """The CPU side of e2e_single_call: T = host-core-count threads, each encoding ONE blob per call with the oracle's SIMD
    port (parity + CRC32 of all shards, one thread per call -- klauspost would split a call over up to 8 goroutines,
    RS/reedsolomon.go:551-557, which changes latency, not the all-cores throughput reported here)."""
    from oracle import pyoracle
    S = shard_size(blob, K)
    n = K + M
    rs = pyoracle.RS(K, M)
    T = len(os.sched_getaffinity(0)) or 1
    rng = np.random.default_rng(1)
    bufs = [rng.integers(0, 256, (1, n, S), dtype=np.uint8) for _ in range(T)]
    crcs = [np.zeros((1, n), dtype=np.uint32) for _ in range(T)]
    lat = [[] for _ in range(T)]
    stop = [False]

    def worker(t):
        while not stop[0]:
            t0 = time.perf_counter()
            rs.encode_batch_simd(bufs[t], S, S, n * S, 1, threads=1, crc_out=crcs[t])
            lat[t].append(time.perf_counter() - t0)

    th = [threading.Thread(target=worker, args=(t,), daemon=True) for t in range(T)]
    t0 = time.perf_counter()
    for x in th:
        x.start()
    time.sleep(seconds)
    stop[0] = True
    for x in th:
        x.join()
    el = time.perf_counter() - t0
    allv = np.sort(np.concatenate([np.asarray(v) for v in lat if v]))
    calls = int(allv.size)
    return {"threads": T, "calls": calls, "stripes_per_s": round(calls / el, 1), "data_GiB_per_s": round(calls * K * S / el / GIB, 3),
            "p50_ms": round(float(allv[calls // 2]) * 1e3, 3), "p99_ms": round(float(allv[min(calls - 1, int(calls * 0.99))]) * 1e3, 3),
            "impl": f"oracle SIMD port ({rs.simd_kind()}), one stripe and one thread per call"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is Go
    (no toolchain here), so this is the oracle's SIMD port on all host cores; rank 0 only."""
    if rank != 0:
        return
    leg = CpuLeg(args.workload, args.cpu_stripes)
    for _ in range(args.warmup):
        leg.one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        leg.one()
    el = time.perf_counter() - t0
    sample_total = leg.sample * leg.REP
    gibs = K * leg.S * sample_total * args.steps / el / GIB
    line = base_line(args, world, gibs, el / args.steps * 1e3)
    line["impl"] = "reference"
    line["n_gpus"] = args.gpus
    line["cpu_baseline"] = {"value": round(gibs, 3), "unit": "GiB/s", "cores": leg.threads, "kind": "port",
                            "sample": f"{sample_total} stripes per step ({leg.sample} distinct, bounded sample of the "
                                      f"config's batch), {leg.describe()}"}
    line["e2e"] = {"value": round(gibs, 3), "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    line["gpu_launches"] = 0
    print(json.dumps(line), flush=True)


def base_line(args, world, value, ms_per_step):
    S = shard_size(BLOB, K)
    name = "rs_12_4_encode_crc32_data_GiB_per_s" if args.workload == "encode" else "rs_12_4_reconstruct_3erasures_data_GiB_per_s"
    return {
        "metric": name, "value": round(value, 3), "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": ("C2: RS(12,4) encode + fused CRC32-IEEE, 4 MiB blobs" if args.workload == "encode"
                                else "C3: RS(12,4) reconstruct, 3 random erasures per stripe, 4 MiB blobs"),
                   "k": K, "m": M, "shard_bytes": S, "stripes_per_gpu": args.stripes, "crc": bool(args.crc),
                   "l2": "inputs (5.7 GB per GPU) larger than the 126 MB L2; no reuse between steps",
                   "parallelism": f"stripes partitioned over {world} GPU(s), no data-path collective"},
    }


# ---------------------------------------------------------------------------------------------------------
# the GPU arm
# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="encode", choices=["encode", "reconstruct"])
    ap.add_argument("--stripes", type=int, default=1024, help="stripes per GPU per step")
    ap.add_argument("--crc", type=int, default=1, help="fused CRC32 in the encode step (C2 asks for it)")
    ap.add_argument("--cpu-stripes", type=int, default=256, help="stripes in the bounded CPU sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--force", type=int, default=0, help="cubeec_debug_force_kernel value (A/B aid, see include/cubeec.h)")
    ap.add_argument("--single-threads", default="64,256,1000", help="caller threads of the e2e_single_call record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import cubefs_b200 as cb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cubefs_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cb.init([local_rank])
    if args.force:
        cb.force_kernel(args.force)

    # coding matrix: built on rank 0, NCCL-broadcast to the other ranks (the only shared state)
    if rank == 0:
        eng0 = cb.RSEngine(K, M)
        rows = torch.from_numpy(eng0.matrix[K:].copy()).to(dev)
    else:
        rows = torch.zeros((M, K), dtype=torch.uint8, device=dev)
    if world > 1:
        dist.broadcast(rows, src=0)
    eng = cb.RSEngine(K, M, parity_rows=rows.cpu().numpy())

    S = shard_size(BLOB, K)
    P = (S + 127) // 128 * 128
    n = K + M
    ns = args.stripes
    g = torch.Generator(device=dev).manual_seed(0xC0BEF5 + rank)
    batch = torch.empty((ns, n, P), dtype=torch.uint8, device=dev)
    for s0 in range(0, ns, 64):
        batch[s0:s0 + 64] = torch.randint(0, 256, batch[s0:s0 + 64].shape, dtype=torch.uint8, device=dev, generator=g)
    dcrc = torch.zeros(ns * n, dtype=torch.int32, device=dev)
    dok = torch.zeros(ns, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    rng = np.random.default_rng(0xC0BEF5 + rank)
    present3 = np.ones((ns, n), dtype=np.uint8)
    for s in range(ns):
        present3[s, rng.choice(n, size=3, replace=False)] = 0
    present1 = np.ones((ns, n), dtype=np.uint8)
    present1[:, 3] = 0   # one broken vuid: the same shard index missing in every stripe (worker_slice_recover.go:822-871)
    sample_ids = sorted({0, ns - 1, *[int(x) for x in rng.choice(ns, size=min(6, ns), replace=False)]})

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def enc(crc=True):
        eng.dev_encode(batch.data_ptr(), S, P, n * P, ns, d_crc=dcrc.data_ptr() if crc else 0, stream=stream, device=local_rank)

    def rec(present):
        eng.dev_reconstruct(batch.data_ptr(), S, P, n * P, ns, present, stream=stream, device=local_rank)

    def ver():
        eng.dev_verify(batch.data_ptr(), S, P, n * P, ns, dok.data_ptr(), stream=stream, device=local_rank)

    def erase(present):
        """overwrite the shards a reconstruct has to regenerate, so a step that did nothing cannot pass the check"""
        rows_, cols_ = np.nonzero(present == 0)
        batch[torch.from_numpy(rows_).to(dev), torch.from_numpy(cols_).to(dev)] = 0xA5

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / steps

    # ---- oracle checks on sampled stripes of the timed batch -------------------------------------------------
    def host_stripe(s):
        return batch[s, :, :S].cpu().numpy()

    def check_encode(with_crc):
        from oracle import pyoracle
        rs = pyoracle.RS(K, M)
        crcs = dcrc.cpu().numpy().view(np.uint32).reshape(ns, n)
        for s in sample_ids:
            h = host_stripe(s)
            want = [h[i].copy() for i in range(K)] + [np.zeros(S, np.uint8) for _ in range(M)]
            rs.encode(want)
            for i in range(K, n):
                if not np.array_equal(h[i], want[i]):
                    raise SystemExit(f"bench check FAILED: parity shard {i} of stripe {s} differs from the oracle")
            if with_crc:
                for i in range(n):
                    if int(crcs[s, i]) != zlib.crc32(want[i].tobytes()):
                        raise SystemExit(f"bench check FAILED: CRC of shard {i} of stripe {s} differs from zlib")
        return len(sample_ids)

    def check_reconstruct(originals, present):
        for s in sample_ids:
            h = host_stripe(s)
            for i in np.nonzero(present[s] == 0)[0]:
                if not np.array_equal(h[i], originals[s][i]):
                    raise SystemExit(f"bench check FAILED: reconstructed shard {i} of stripe {s} differs from the original")
        return len(sample_ids)

    def last_step_outputs():
        """What a caller of the timed path receives, for the checked stripes (bytes as float32, CRCs as float64: exact)."""
        out = {"stripe_ids": np.asarray(sample_ids, dtype=np.float64)}
        if args.workload == "reconstruct":
            lost = [np.nonzero(present3[s] == 0)[0] for s in sample_ids]
            out["erased_shards"] = np.asarray(lost, dtype=np.float64)
            out["reconstructed"] = np.stack([host_stripe(s)[i] for s, i in zip(sample_ids, lost)]).astype(np.float32)
        else:
            out["parity"] = np.stack([host_stripe(s)[K:] for s in sample_ids]).astype(np.float32)
            if args.crc:
                out["crc32"] = dcrc.cpu().numpy().view(np.uint32).reshape(ns, n).astype(np.float64)
        return out

    # ---- headline -------------------------------------------------------------------------------------------
    peak, peak_src = measured_peak()
    enc(True)
    barrier()
    originals = None if args.no_check else {s: host_stripe(s) for s in sample_ids}   # encoded stripes (oracle-checked below)
    erasures = 0
    if args.workload == "reconstruct":
        erase(present3)
        erasures = 3
        step = lambda: rec(present3)   # noqa: E731
    else:
        step = lambda: enc(bool(args.crc))   # noqa: E731
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = cb.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    tw0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    tw1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    launches = cb.kernel_launches() - launches0
    head_kernel = cb.last_kernel()
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = K * S * ns * world / (ms_step * 1e-3) / GIB
    checked = 0
    if not args.no_check:
        checked = check_reconstruct(originals, present3) if args.workload == "reconstruct" else check_encode(bool(args.crc))
    if args.dump_outputs and rank == 0:   # before the extra records below run other kernels over the same batch
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in last_step_outputs().items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    def record(ms_, alg_bytes, kernel):
        ach = alg_bytes / (ms_ * 1e-3) / 1e9
        return {"ms": round(ms_, 4), "data_GiB_per_s": round(K * S * ns / (ms_ * 1e-3) / GIB, 1), "achieved_GBps": round(ach, 1),
                "frac": round(ach / peak, 4), "frac_nominal_8TBs": round(ach / NOMINAL_HBM_GBS, 4), "kernel": kernel,
                "algorithmic_bytes": alg_bytes}

    # ---- the rest of "encode + reconstruct": plain encode, verify, C3, single-pattern repair (N = 1 only) ----------
    extra = None
    if world == 1 and not args.no_extra:
        extra = {}
        st, wu = args.steps, 3
        if args.workload == "reconstruct":
            rec(present3)   # leave the batch consistent
        ms_ = timed(lambda: enc(False), st, wu)
        extra["encode_nocrc"] = record(ms_, n * S * ns, cb.last_kernel())
        ms_ = timed(lambda: enc(True), st, wu)
        extra["encode_crc"] = record(ms_, n * S * ns, cb.last_kernel())
        ms_ = timed(ver, st, wu)
        extra["verify"] = record(ms_, n * S * ns, cb.last_kernel())
        if not args.no_check and int(dok.sum().item()) != ns:
            raise SystemExit("bench check FAILED: dev_verify rejects a stripe the engine just encoded")
        # the shard checksums on their own (what a blobnode does on read / inspect, and the replica modes on write)
        from cubefs_b200.engine import dev_crc32
        dcrc2 = torch.zeros_like(dcrc)
        ms_ = timed(lambda: dev_crc32(batch.data_ptr(), S, P, ns * n, d_whole=dcrc2.data_ptr(), stream=stream, device=local_rank), st, wu)
        extra["crc32_shards"] = record(ms_, n * S * ns, cb.last_kernel())
        if not args.no_check:
            if not torch.equal(dcrc2, dcrc):
                raise SystemExit("bench check FAILED: stand-alone shard CRCs differ from the fused kernel's")
            extra["crc32_shards"]["checked_shards"] = int(ns * n)
        for name, pres, e in (("reconstruct_3e", present3, 3), ("reconstruct_1pattern", present1, 1)):
            erase(pres)
            ms_ = timed(lambda pres=pres: rec(pres), st, wu)
            extra[name] = record(ms_, (K + e) * S * ns, cb.last_kernel())
            extra[name]["patterns"] = int(len({bytes(r) for r in pres}))
            if not args.no_check:
                extra[name]["checked_stripes"] = check_reconstruct(originals, pres)
        extra["note"] = (f"same 1024-stripe batch, {st} timed steps after {wu} warm-up each, CUDA events; reconstruct regenerates "
                         "shards that were overwritten with 0xA5 first; algorithmic bytes: encode/verify (k+m)*S, reconstruct (k+e)*S")

    # ---- end to end through the host entry points (pinned host buffers; then single-stripe pageable calls) ----
    e2e = None
    e2e_single = None
    if not args.no_e2e and args.workload == "encode":
        del batch
        torch.cuda.empty_cache()
        ns_e = min(ns, 512)
        host = torch.empty((ns_e, n * S), dtype=torch.uint8).pin_memory()
        host.copy_(torch.randint(0, 256, host.shape, dtype=torch.uint8))
        hnp = host.numpy()
        for _ in range(2):
            crc_h, _ = eng.encode_contig(hnp, S, ns_e, n * S, crc=bool(args.crc))
        barrier()
        t0 = time.perf_counter()
        reps = args.steps
        for _ in range(reps):
            eng.encode_contig(hnp, S, ns_e, n * S, crc=bool(args.crc))
        torch.cuda.synchronize(dev)
        el = time.perf_counter() - t0
        t = torch.tensor([el], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el = float(t.item())
        e2e = {"value": round(K * S * ns_e * world * reps / el / GIB, 3), "unit": "GiB/s",
               "h2d_bytes_per_step": K * S * ns_e, "d2h_bytes_per_step": M * S * ns_e + (n * ns_e * 4 if args.crc else 0),
               "stripes_per_step": ns_e, "numa": numa,
               "api": "cubeec_encode_contig (pinned host ec.Buffer layout, H2D+kernel+D2H pipelined)"}
        if not args.no_check:
            from oracle import pyoracle
            rs = pyoracle.RS(K, M)
            for s in (0, ns_e - 1):
                row = hnp[s].reshape(n, S)
                want = [row[i].copy() for i in range(K)] + [np.zeros(S, np.uint8) for _ in range(M)]
                rs.encode(want)
                ok = all(np.array_equal(row[i], want[i]) for i in range(n))
                ok = ok and (crc_h is None or all(int(crc_h[s, i]) == zlib.crc32(want[i].tobytes()) for i in range(n)))
                if not ok:
                    raise SystemExit(f"bench check FAILED: e2e stripe {s} differs from the oracle")
            e2e["checked_stripes"] = 2
        if world == 1 and hasattr(eng, "encode_single_call_bench"):
            e2e_single = eng.encode_single_call_bench(BLOB, [int(x) for x in args.single_threads.split(",")],
                                                      check=not args.no_check)
            if not args.no_cpu:
                e2e_single["cpu_same_call_shape"] = cpu_single_call(BLOB)

    if rank == 0:
        alg = ((K + M) if args.workload == "encode" else (K + erasures)) * S * ns
        achieved = alg / (ms_step * 1e-3) / 1e9
        line = base_line(args, world, value, ms_step)
        line["clocks"] = clocks
        line["gpu_launches"] = int(launches)
        line["kernel"] = head_kernel
        line["checked_stripes"] = checked
        traffic, traffic_src = traffic_from_profile(head_kernel, ns)
        line["roofline"] = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                            "frac": round(achieved / peak, 4), "frac_nominal_8TBs": round(achieved / NOMINAL_HBM_GBS, 4),
                            "traffic": traffic, "traffic_from_profile": traffic_src, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": alg,
                            "note": "per-GPU figure; device time of one step (coding kernel + CRC finalize) by CUDA events; "
                                    "traffic is read from the committed ncu summary named in traffic_from_profile, not measured in this run"}
        line["extra"] = extra
        line["e2e"] = e2e
        line["e2e_single_call"] = e2e_single
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args.workload, args.cpu_stripes)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
