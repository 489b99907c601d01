#!/usr/bin/env python
"""bench.py -- the BASELINE.json metric: uncompressed GB/s of LZ4_decompress_safe over a stream of
independent 64 KB blocks (tests/datagen P50), per GPU count, against the HBM roofline.

    python bench.py [--gpus N --steps K --warmup W]          our CUDA path
    python bench.py --impl reference [...]                    the reference's CPU implementation
    torchrun --nproc-per-node N bench.py --gpus N ...         one rank per GPU (weak scaling)
    python bench.py [...] --dump-outputs DIR                  + what the last timed step decoded, as DIR/*.npy

One "step" = one pass of the hot path (scan + expand kernels) over this rank's whole batch
(default 4 GiB = 65 536 blocks per GPU).  Inputs are device resident for `value`; `e2e` runs the
same workload through LZ4B200_decompress_blocks_host with pinned HOST buffers (H2D and D2H copies
inside the timed region).  Prints ONE JSON line (rank 0).
"""
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
SEG = 64 << 20                      # datagen segment: RDG_genBuffer(64 MiB, P, seed) (SURVEY 8d C2)
METRIC = "uncompressed GB/s, LZ4_decompress_safe over independent 64 KB blocks (datagen P50)"
GB = 1e9


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gib", type=float, default=4.0, help="uncompressed GiB per GPU")
    ap.add_argument("--proba", type=float, default=0.5, help="datagen match probability (P50)")
    ap.add_argument("--accel", type=int, default=1)
    ap.add_argument("--block-kb", type=int, default=64, help="block size in KB (64 = BASELINE configs 1-3; 4096 = lz4frame 4 MB blocks)")
    ap.add_argument("--ref-gib", type=float, default=1.0, help="--impl reference: GiB of the workload each step decodes (bounded sample)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--chunks", type=int, default=1, help="N > 1: pieces of a rank's shard whose exchange overlaps the decode of the next piece")
    ap.add_argument("--ceiling", action="store_true",
                    help="also time the rows kernel's skeleton without the decode (TMA in/out only; + one LDS/STS per output byte)")
    ap.add_argument("--exchange", default="nccl", choices=["peer", "nccl"],
                    help="N > 1: 'nccl' = grouped NCCL send/recv per chunk, 'peer' = copy-engine pushes into the peers' frames (CUDA IPC)")
    ap.add_argument("--reserve-sms", type=int, default=0,
                    help="N > 1: SMs the persistent decode kernels leave to the concurrent exchange kernels (LZ4B200_RESERVE_SMS)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step decoded to DIR/*.npy (a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# --------------------------------------------------------------------------------------------
# --dump-outputs: the decoded frame of the last timed step, so that two builds can be compared output for output
# --------------------------------------------------------------------------------------------
DUMP_DECODED_BYTES = 4 << 20        # decoded bytes sampled into decoded_blocks.npy (16 MiB as float32)
DUMP_MAX_SIZES = 1 << 21            # per-block return values written in full up to this many blocks, else a sample


def dump_outputs(dirname, n_blocks, block_rows, sizes):
    """Write decoded_blocks.npy (float32: the bytes of whole blocks picked with a fixed seed, at most
    DUMP_DECODED_BYTES in all), decoded_block_ids.npy (their indices) and decoded_sizes.npy (the return value of
    every block; beyond DUMP_MAX_SIZES blocks a seeded sample, with decoded_sizes_ids.npy).  block_rows(ids) gives
    the decoded bytes of blocks `ids` as a (len(ids), >= width) uint8 array; sizes is the int array of all returns.
    The same arguments give the same blocks, and the dump stays below 64 MB whatever the workload size."""
    os.makedirs(dirname, exist_ok=True)

    def pick(k):
        if n_blocks <= k:
            return np.arange(n_blocks)
        return np.sort(np.random.default_rng(0).choice(n_blocks, k, replace=False))

    width = min(BLOCK, DUMP_DECODED_BYTES)
    ids = pick(max(1, DUMP_DECODED_BYTES // BLOCK))
    np.save(os.path.join(dirname, "decoded_block_ids.npy"), ids.astype(np.float64))
    np.save(os.path.join(dirname, "decoded_blocks.npy"), np.asarray(block_rows(ids))[:, :width].astype(np.float32))
    ids = pick(DUMP_MAX_SIZES)
    if len(ids) < n_blocks:
        np.save(os.path.join(dirname, "decoded_sizes_ids.npy"), ids.astype(np.float64))
    np.save(os.path.join(dirname, "decoded_sizes.npy"), np.asarray(sizes)[ids].astype(np.float64))


# --------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for k, nme in enumerate(names):
                if len(f) > 3 + k and f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation, all host threads
# --------------------------------------------------------------------------------------------
def cpu_codec():
    """(codec, kind): the compiled reference (oracle/_ref) when present, else the oracle port."""
    from oracle.pyoracle import Oracle, Reference, have_reference
    orc = Oracle()
    if have_reference():
        return orc, Reference(), "reference"
    return orc, orc, "port"


def cpu_decompress_rate(orc, codec, comp, offs, sizes, n_blocks, threads, passes):
    out = np.empty(n_blocks * BLOCK, dtype=np.uint8)
    best = None
    for _ in range(passes):
        t, rets = orc.time_decompress(codec, comp, offs, sizes, out, BLOCK, threads)
        assert t > 0 and (rets == BLOCK).all(), "CPU reference failed to decode"
        best = t if best is None else min(best, t)
    return n_blocks * BLOCK / best / GB, out


def run_reference(args):
    """The reference's own CPU implementation (oracle/_ref when it was compiled, else the oracle port) on this box's
    host cores: all threads, one pinned worker per CPU, static block partition (programs/bench.c:464-555 loops one
    thread the same way), every buffer first-touched by the worker that uses it, compressed input packed like
    the GPU arm's.  `value` comes from the MEDIAN step (robust against a disturbed pass); best and mean are
    reported beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    orc, codec, kind = cpu_codec()
    cores = len(os.sched_getaffinity(0)) or os.cpu_count() or 1
    # a BOUNDED sample of the workload: the first GiB of the same stream (same generator, seeds, block size).  Measured on
    # the driver's boxes (profiles/): over 4 GiB the same code runs 2-4x slower and unstable on a shared host, over 1 GiB it
    # reproduces within a few percent -- and the faster figure is the one a CPU baseline should be given.
    gib = min(args.gib, args.ref_gib)
    n_blocks = int(gib * (1 << 30)) // BLOCK
    data = np.empty(n_blocks * BLOCK, dtype=np.uint8)
    orc.first_touch(data, BLOCK, n_blocks, cores)
    orc.datagen_mt(n_blocks * BLOCK, SEG, args.proba, 0, cores, out=data)
    cap = orc.compress_bound(BLOCK)
    stride = (cap + 15) // 16 * 16
    slots = np.empty(n_blocks * stride, dtype=np.uint8)
    orc.first_touch(slots, stride, n_blocks, cores)
    tcs = []
    for _ in range(3):
        tc, csz = orc.time_compress(codec, data, BLOCK, slots, stride, args.accel, cores)
        assert tc > 0
        tcs.append(tc)
    offs = np.zeros(n_blocks + 1, dtype=np.int64)
    np.cumsum(csz, out=offs[1:])
    packed = np.empty(int(offs[-1]) + 16, dtype=np.uint8)
    orc.pack(slots, stride, csz, offs[:-1].copy(), packed, cores)       # the GPU arm decodes a packed stream too
    del slots
    offs = offs[:-1].copy()
    out = np.empty(n_blocks * BLOCK, dtype=np.uint8)
    orc.first_touch(out, BLOCK, n_blocks, cores)
    t1, _ = orc.time_decompress(codec, packed, offs[:min(n_blocks, 2048)], csz[:min(n_blocks, 2048)], out, BLOCK, 1)
    single = min(n_blocks, 2048) * BLOCK / t1 / GB
    for _ in range(max(args.warmup, 1)):
        orc.time_decompress(codec, packed, offs, csz, out, BLOCK, cores)
    times = []
    for _ in range(args.steps):
        t, rets = orc.time_decompress(codec, packed, offs, csz, out, BLOCK, cores)
        assert t > 0 and (rets == BLOCK).all()
        times.append(t)
    assert (out == data).all(), "reference round trip mismatch"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n_blocks, lambda ids: out.reshape(n_blocks, BLOCK)[ids], rets)
    med, best, mean = float(np.median(times)), min(times), sum(times) / len(times)
    nbytes = n_blocks * BLOCK
    value = nbytes / med / GB
    sample = "the first %d blocks of %d KB (%.2f GiB) of the workload, datagen P%d, %d pinned host threads (one per CPU), static partition, packed input" % (
        n_blocks, BLOCK // 1024, nbytes / (1 << 30), round(args.proba * 100), cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": round(1e3 * med, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(int(args.gib * (1 << 30)) // BLOCK, args.gib, args.proba, args.accel, nbytes / float(csz.sum()), args.gpus),
        "timing": {"value_from": "median step", "best_GBps": round(nbytes / best / GB, 3),
                   "median_GBps": round(value, 3), "mean_GBps": round(nbytes / mean / GB, 3),
                   "spread": round(max(times) / best, 3)},
        "cpu_baseline": {"value": round(value, 3), "unit": "GB/s", "cores": cores, "kind": kind, "sample": sample,
                         "single_thread_GBps": round(single, 3),
                         "compress_GBps_all_threads": round(nbytes / min(tcs) / GB, 3)},
        "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if max(times) / best > 1.5:
        line["warning"] = "reference passes disagree by more than 1.5x (%.1f .. %.1f GB/s): the host was disturbed" % (
            nbytes / max(times) / GB, nbytes / best / GB)
    print(json.dumps(line))
    return 0


def workload_config(n_blocks, gib, proba, accel, ratio, gpus):
    """`config` of the JSON line: identical for both arms (the driver compares it)."""
    return {"workload": "decompress-only, %d independent %d KB blocks per GPU (%.2f GiB), tests/datagen P%d "
                        "(RDG_genBuffer per 64 MiB segment, seed=rank*64+k), compressed by LZ4_compress_fast accel %d"
                        % (n_blocks, BLOCK // 1024, gib, round(proba * 100), accel),
            "block_bytes": BLOCK, "blocks_per_gpu": n_blocks, "ratio": round(ratio, 2),
            "l2": "the inputs of a step (%.1f GiB compressed + %.1f GiB decoded) exceed the 126 MB L2 and every CPU cache; no flush needed"
                  % (n_blocks * BLOCK / ratio / (1 << 30), n_blocks * BLOCK / (1 << 30)),
            "parallelism": "blocks partitioned contiguously over %d rank(s); for N > 1 the timed step ends with the exchange "
                           "of the decoded shards (every rank holds the whole frame; --chunks > 1 overlaps it piecewise with the decode)"
                           % gpus}


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(torch, local):
    """Host-side tuning for the e2e leg: run (and first-touch / pin host buffers) on the CPU cores of
    the NUMA node the GPU hangs off, so pinned-memory PCIe copies do not cross the socket link."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids)
        return {"numa_node": node, "cpus": len(ids)}
    except Exception:
        return None


def pcie_probe(torch, device, nbytes=1 << 30):
    """Plain pinned-memory copy rates (GB/s) on this box: the ceiling of any host-buffer path."""
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device=device)
    res = {}
    for name, dst, src in (("h2d", d, h), ("d2h", h, d)):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        res[name] = round(3 * nbytes / (time.perf_counter() - t0) / GB, 2)
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from lz4_b200 import _lib, batch
    from lz4_b200 import dist as ldist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    lib = _lib.load()
    assert lib.LZ4B200_device_count() > 0, "bench.py needs a CUDA device (no CPU fallback)"

    from oracle.pyoracle import Oracle          # input generator + checker + cpu_baseline only
    orc = Oracle()
    cores = os.cpu_count() or 1
    n_blocks = int(args.gib * (1 << 30)) // BLOCK
    total = n_blocks * BLOCK
    seed0 = rank * 64                           # SURVEY 8(d) C4: seed = rank*64 + k
    host = orc.datagen_mt(total, SEG, args.proba, seed0, max(1, cores // world))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_source = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)"

    def barrier():
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)

    # ---- compress leg (BASELINE config 3): ON THE GPU, byte-identical to the reference; timed with its own clocks ----
    src = torch.from_numpy(host).to(device)
    slots, csizes, stride = batch.compress_blocks(src, BLOCK, args.accel)      # warm-up + result
    torch.cuda.synchronize()
    KC = max(1, min(args.steps, 3))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tc0 = time.time()
    ev0.record()
    for _ in range(KC):
        batch.compress_blocks(src, BLOCK, args.accel, slots=slots, out_sizes=csizes)
    ev1.record()
    torch.cuda.synchronize()
    tc1 = time.time()
    compress_ms = ev0.elapsed_time(ev1) / KC
    compress_clocks = sampler.summary(tc0, tc1)
    # the parallel-parse compressor (throughput mode): valid LZ4, deterministic, not byte-identical; same clocks rule
    pslots = torch.empty_like(slots)
    psizes = torch.empty_like(csizes)
    batch.compress_blocks(src, BLOCK, args.accel, slots=pslots, out_sizes=psizes, mode="parallel")
    torch.cuda.synchronize()
    tp0 = time.time()
    ev0.record()
    for _ in range(KC):
        batch.compress_blocks(src, BLOCK, args.accel, slots=pslots, out_sizes=psizes, mode="parallel")
    ev1.record()
    torch.cuda.synchronize()
    tp1 = time.time()
    par_ms = ev0.elapsed_time(ev1) / KC
    par_clocks = sampler.summary(tp0, tp1)
    psz_host = psizes.cpu().numpy()
    par_bytes = int(psz_host.sum())
    for i in np.random.default_rng(100 + rank).integers(0, n_blocks, 8):     # checker: the ORACLE's decoder expands it to the input
        blk = pslots[i * stride:i * stride + int(psz_host[i])].cpu().numpy().tobytes()
        dret, dout = orc.decompress(blk, BLOCK)
        assert dret == BLOCK and dout == host[i * BLOCK:(i + 1) * BLOCK].tobytes(), "parallel compressor: block %d does not round-trip" % i
    del pslots
    packed, offs_all = batch.pack_blocks(slots, stride, csizes)
    offs = offs_all[:-1].contiguous()
    torch.cuda.synchronize()
    comp_bytes = int(offs_all[-1].item())
    csz_host = csizes.cpu().numpy()
    # checker: a sample of GPU-compressed blocks must equal the oracle's bytes
    rng = np.random.default_rng(rank)
    for i in rng.integers(0, n_blocks, 8):
        eret, eout = orc.compress(host[i * BLOCK:(i + 1) * BLOCK], args.accel)
        got = slots[i * stride:i * stride + int(csz_host[i])].cpu().numpy().tobytes()
        assert int(csz_host[i]) == eret and got == eout, "GPU compressor differs from the oracle at block %d" % i
    packed = packed[:comp_bytes + 16].clone()
    del slots
    torch.cuda.empty_cache()

    # decoded frame: every rank decodes INTO ITS SLICE of the full buffer (N > 1: the exchange fills the rest)
    full = torch.empty(world * total, dtype=torch.uint8, device=device)
    out = full[rank * total:(rank + 1) * total]
    rets = torch.empty(n_blocks, dtype=torch.int32, device=device)
    ws = torch.empty(int(lib.LZ4B200_decompress_workspace_bytes_for(n_blocks, 0, BLOCK)), dtype=torch.uint8, device=device)

    def decode(lo=0, hi=n_blocks, phases=3):
        batch.decompress_blocks(packed, offs[lo:hi], csizes[lo:hi], BLOCK, out=out[lo * BLOCK:hi * BLOCK],
                                out_sizes=rets[lo:hi], workspace=ws, phases=phases)

    peer, exchange = None, args.exchange
    if world > 1 and exchange == "peer":
        # every rank must take the same path: agree on whether the peers' frames could be mapped (CUDA IPC + peer access)
        try:
            peer = ldist.PeerFrame(full)
            ok = 1
        except Exception as e:                     # noqa: BLE001 -- any failure means "use NCCL instead", on every rank
            sys.stderr.write("rank %d: peer-memory exchange unavailable (%s); falling back to NCCL send/recv\n" % (rank, e))
            ok = 0
        t = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 0:
            peer, exchange = None, "nccl"

    def step():
        """one pass of the hot path over this rank's batch; N > 1: + the exchange of the decoded shards, overlapped"""
        if world == 1:
            decode()
        else:
            ldist.decode_and_allgather(full, n_blocks, BLOCK, decode, n_chunks=args.chunks, peer=peer)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    assert bool((rets == BLOCK).all()) and torch.equal(out, src), "GPU decode mismatch"
    gather_ok = None
    if world > 1:                               # every rank's shard arrived: compare against regenerated neighbours
        nb = (rank + 1) % world
        other = orc.datagen_mt(SEG, SEG, args.proba, nb * 64, max(1, cores // world))
        gather_ok = bool(torch.equal(full[nb * total:nb * total + SEG].cpu(), torch.from_numpy(other)))
        assert gather_ok, "exchanged frame differs from the neighbour's data"

    # ---- timed region: K steps, device resident, CUDA events on the launching stream ----
    K = args.steps
    launches0 = lib.LZ4B200_launch_count()
    barrier(); torch.cuda.synchronize()
    t_wall0 = time.time()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for k in range(K):
        step()
    end.record()
    torch.cuda.synchronize(); barrier()
    t_wall1 = time.time()
    launches = lib.LZ4B200_launch_count() - launches0
    my_ms = start.elapsed_time(end)
    elapsed_ms = my_ms
    per_rank_ms = None
    if world > 1:
        t = torch.zeros(world, dtype=torch.float64, device=device)
        t[rank] = my_ms
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        per_rank_ms = [round(float(x) / K, 4) for x in t.tolist()]
        elapsed_ms = float(t.max().item())
    value = world * total * K / (elapsed_ms * 1e-3) / GB
    clocks = sampler.summary(t_wall0, t_wall1)
    if args.dump_outputs:                       # before the phase timing below decodes again into the same frame
        all_rets = rets
        if world > 1:
            all_rets = torch.empty(world * n_blocks, dtype=torch.int32, device=device)
            dist.all_gather_into_tensor(all_rets, rets)
        if rank == 0:
            width = min(BLOCK, DUMP_DECODED_BYTES)
            dump_outputs(args.dump_outputs, world * n_blocks,
                         lambda ids: full.view(-1, BLOCK)[torch.from_numpy(ids).to(device), :width].cpu().numpy(),
                         all_rets.cpu().numpy())

    # ---- the two kernels of the decode, timed separately (same launches, events between the phases) ----
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    barrier(); torch.cuda.synchronize()
    for k in range(K):
        evs[k][0].record()
        decode(phases=1)             # scan kernel
        evs[k][1].record()
        decode(phases=2)             # expand kernel (dominant)
        evs[k][2].record()
    torch.cuda.synchronize()
    scan_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / K
    expand_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / K
    codec_ms = sum(e[0].elapsed_time(e[2]) for e in evs) / K
    if world > 1:
        t = torch.tensor([codec_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        codec_ms_max = float(t.item())
    else:
        codec_ms_max = codec_ms

    # ---- ceiling of the rows kernel's structure: the same persistent TMA-in -> smem -> TMA-out skeleton, no decode ----
    ceiling = None
    if args.ceiling and BLOCK == 65536:
        import ctypes as C
        fn = lib.LZ4B200_debug_ceiling
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p]
        st = torch.cuda.current_stream().cuda_stream
        ceiling = {"what": "lz4_ceiling_kernel: one CTA per SM, TMA bulk load of each compressed block, TMA bulk store of 64 KB, "
                           "same batch; the bytes written are meaningless"}
        for mode, key in ((0, "tma_only"), (1, "tma_plus_one_lds_sts_per_byte")):
            for _ in range(2):
                assert fn(packed.data_ptr(), offs.data_ptr(), csizes.data_ptr(), out.data_ptr(), BLOCK, n_blocks, mode, st) == 0
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                fn(packed.data_ptr(), offs.data_ptr(), csizes.data_ptr(), out.data_ptr(), BLOCK, n_blocks, mode, st)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / K
            ceiling[key] = {"ms": round(ms, 4), "GBps_algorithmic": round((comp_bytes + total) / (ms * 1e-3) / GB, 1)}
        decode()                                             # restore the decoded bytes
        torch.cuda.synchronize()

    # ---- e2e: same workload through the host-buffer C-ABI call, pinned host memory ----
    e2e = None
    if not args.no_e2e:
        all_cpus = os.sched_getaffinity(0)
        numa = bind_to_gpu_numa_node(torch, local)      # pin + first-touch the host buffers next to the GPU
        h_comp = torch.empty(comp_bytes + 16, dtype=torch.uint8, pin_memory=True)
        h_comp.copy_(packed[:comp_bytes + 16])
        h_offs = offs.cpu().numpy()
        h_out = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        h_rets = np.zeros(n_blocks, dtype=np.int32)

        def e2e_step():
            rc = lib.LZ4B200_decompress_blocks_host(h_comp.data_ptr(), h_offs.ctypes.data, csz_host.ctypes.data,
                                                    h_out.data_ptr(), BLOCK, BLOCK, h_rets.ctypes.data, n_blocks)
            _lib.check(rc, "LZ4B200_decompress_blocks_host")

        e2e_step()
        assert (h_rets == BLOCK).all() and bool((h_out.numpy() == host).all()), "e2e decode mismatch"
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        t1 = time.perf_counter()
        dt = t1 - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        pcie = pcie_probe(torch, device)
        e2e = {"value": round(world * total * args.e2e_steps / dt / GB, 3), "unit": "GB/s",
               "pcie_pinned_copy_GBps": pcie, "host_numa_binding": numa,
               "h2d_bytes_per_step": int(comp_bytes + n_blocks * 12), "d2h_bytes_per_step": int(total + n_blocks * 4),
               "steps": args.e2e_steps, "api": "LZ4B200_decompress_blocks_host (pinned host buffers)",
               "ceiling": "PCIe: %.1f GB of output per step cannot leave the GPU faster than the pinned D2H rate (%.1f GB/s), "
                          "so e2e <= that rate whatever the kernels do" % (total / GB, pcie["d2h"])}
        del h_comp, h_out
        os.sched_setaffinity(0, all_cpus)
    sampler.stop()

    # ---- compressed-side reassembly on NCCL (N > 1): size table + padded shards, verified ----
    comp_gather = None
    if world > 1:
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ldist.allgather_compressed(packed, comp_bytes, csizes)
        torch.cuda.synchronize(); barrier()
        g0.record()
        all_sizes, shards, shard_bytes = ldist.allgather_compressed(packed, comp_bytes, csizes)
        g1.record()
        torch.cuda.synchronize()
        ok = bool(torch.equal(all_sizes[rank * n_blocks:(rank + 1) * n_blocks], csizes)) and \
            bool(torch.equal(shards[rank, :comp_bytes], packed[:comp_bytes])) and int(shard_bytes[rank]) == comp_bytes
        t = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        comp_gather = {"ms": round(float(t.item()), 3), "bytes_in_per_rank": int(shard_bytes.sum().item()) - comp_bytes,
                       "verified": ok}
        del shards

    # ---- cpu baseline (rank 0, N == 1): the reference's CPU path on a bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        _, codec, kind = cpu_codec()
        nb = min(n_blocks, max(1, (1 << 30) // BLOCK))
        hi = int(offs_all[nb].item())
        comp_host = packed[:hi + 16].cpu().numpy()
        offs_host = offs[:nb].cpu().numpy()
        sizes_host = csz_host[:nb].copy()
        one, dec = cpu_decompress_rate(orc, codec, comp_host, offs_host, sizes_host, nb, 1, 2)
        assert (dec == host[:nb * BLOCK]).all()
        allc, _ = cpu_decompress_rate(orc, codec, comp_host, offs_host, sizes_host, nb, cores, 5)
        cpu = {"value": round(allc, 3), "unit": "GB/s", "cores": cores, "kind": kind,
               "sample": "first %d blocks (%.2f GiB) of the same stream, best of 5 passes, %d threads" % (
                   nb, nb * BLOCK / (1 << 30), cores),
               "single_thread_GBps": round(one, 3)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    algo_bytes = comp_bytes + total                      # C_i read once + U_i written once (SURVEY 8d)
    achieved = algo_bytes / (expand_ms * 1e-3) / GB
    step_achieved = algo_bytes / (codec_ms * 1e-3) / GB
    traffic, step_traffic, traffic_src = None, None, None
    try:                                                 # ncu --set full captures, summarised per 64 KB block by profiles/summarize.py
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if abs(args.proba - tj.get("proba", 0.5)) < 1e-9 and BLOCK == tj.get("block_bytes", 65536):
            traffic = int(tj["expand_dram_bytes_per_block"] * n_blocks)
            step_traffic = int((tj["expand_dram_bytes_per_block"] + tj["scan_dram_bytes_per_block"]) * n_blocks)
            traffic_src = "profiles/traffic.json: " + "; ".join("%s = %s" % kv for kv in sorted(tj.get("sources", {}).items()) if kv[0] in ("expand", "scan"))
    except (OSError, ValueError, KeyError):
        pass
    config = workload_config(n_blocks, args.gib, args.proba, args.accel, total / comp_bytes, world)
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": K,
        "warmup": max(args.warmup, 3), "ms_per_step": round(elapsed_ms / K, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config,
        "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic,
                     "kernel": "lz4_expand_rows_kernel", "kernel_ms": round(expand_ms, 4), "scan_kernel_ms": round(scan_ms, 4),
                     "algorithmic_bytes_per_launch": algo_bytes,
                     "step": {"kernels": "lz4_scan_kernel + lz4_expand_rows_kernel (+ the empty generic expand launch)",
                              "ms": round(codec_ms, 4), "achieved": round(step_achieved, 2),
                              "frac": round(step_achieved / peak, 4), "traffic": step_traffic},
                     "traffic_source": traffic_src,
                     "peak_source": peak_source, **({"ceiling": ceiling} if ceiling else {})},
        "clocks": clocks,
        "gpu_launches": int(launches),
        "compress": {"GBps": round(total / (compress_ms * 1e-3) / GB, 3), "ms": round(compress_ms, 3),
                     "ratio": round(total / comp_bytes, 4), "accel": args.accel, "steps": KC,
                     "kernel": "lz4_encode_kernel (byte-identical to LZ4_compress_fast; sample checked against the oracle)",
                     "roofline": {"bound": "hbm", "achieved": round(algo_bytes / (compress_ms * 1e-3) / GB, 2), "peak": peak,
                                  "unit": "GB/s", "frac": round(algo_bytes / (compress_ms * 1e-3) / GB / peak, 4)},
                     "clocks": compress_clocks},
        "compress_parallel": {"GBps": round(total / (par_ms * 1e-3) / GB, 3), "ms": round(par_ms, 3),
                              "ratio": round(total / par_bytes, 4), "ratio_vs_reference": round(comp_bytes / par_bytes, 4),
                              "accel": args.accel, "steps": KC,
                              "kernel": "lz4_encode_par_kernel (valid LZ4, deterministic, NOT byte-identical; sample decoded by the oracle)",
                              "roofline": {"bound": "hbm", "achieved": round((total + par_bytes) / (par_ms * 1e-3) / GB, 2), "peak": peak,
                                           "unit": "GB/s", "frac": round((total + par_bytes) / (par_ms * 1e-3) / GB / peak, 4)},
                              "clocks": par_clocks},
    }
    if world > 1:
        how = ("copy-engine pushes into the peers' frames over NVLink peer memory (CUDA IPC), one stream per peer"
               if exchange == "peer" else "grouped NCCL send/recv per chunk")
        line["multi_gpu"] = {"value_includes": "decode + exchange of the decoded shards (%s; %d chunks, exchange of chunk k "
                                               "overlaps the decode of chunk k+1)" % (how, args.chunks),
                             "exchange": exchange, "chunks": args.chunks, "reserve_sms": args.reserve_sms,
                             "per_rank_ms_per_step": per_rank_ms,
                             "codec_only": {"ms_per_step_max_over_ranks": round(codec_ms_max, 4),
                                            "GBps": round(world * total / (codec_ms_max * 1e-3) / GB, 3)},
                             "exchange_bytes_in_per_rank": int((world - 1) * total), "exchange_verified": gather_ok,
                             "compressed_reassembly": comp_gather}
    if e2e:
        line["e2e"] = e2e
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    global BLOCK, METRIC
    args = parse_args()
    if args.reserve_sms > 0:
        os.environ["LZ4B200_RESERVE_SMS"] = str(args.reserve_sms)          # read once by the library's first decode launch
    if args.block_kb != 64:
        BLOCK = args.block_kb * 1024
        METRIC = METRIC.replace("64 KB", "%d KB" % args.block_kb)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
