#!/usr/bin/env python3
"""bench.py — blob hash-and-cache throughput (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic blobs.

  value     whole-job GB/s with the blobs already resident in HBM: one fused
            multi-buffer SHA-256 pass (dm_ingest_device) that reads every byte
            once, advances its blob's digest and writes it into the CAS.
  e2e       the same blobs pushed from HOST memory through the C-ABI the proxy
            would call (dm_proxy_drive -> dm_stream_open/write/finish): ring
            memcpy, H2D DMA, hash, digest read-back, all inside the timed region.
  roofline  the SHA-256 kernel: algorithmic bytes (2 B per blob byte for
            hash-and-cache) / CUDA-event kernel time, against the measured HBM
            copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline / --impl reference
            the hash-and-cache loop north_star attributes to the reference,
            timed on this box's host cores (oracle/cpu_baseline.c: OpenSSL
            EVP_sha256 + memcpy, a stand-in for Go crypto/sha256 — Go is not
            installed and the reference holds no such loop, SURVEY.md §0).

Multi-GPU: one process per GPU under torchrun; blobs are partitioned by the
production routing function (URL-hash for blobs whose digest is not known up
front), per-GPU work is fixed (weak scaling), no data-path collective.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 0xDE40DE1
METRIC = "blob hash-and-cache throughput"
UNIT = "GB/s"

WORKLOADS = {
    # BASELINE.json configs[2]: 256 concurrent 64 MB HF LFS range streams on 1 B200
    "hf_lfs_256x64MiB": {"sizes": [64 << 20] * 256, "baseline_config": 2},
    # BASELINE.json configs[1]: Llama-3-8B safetensors shard set (real shard sizes, SURVEY.md §8d)
    "llama3_8b_shards": {"sizes": [4976698672, 4999802720, 4915916176, 1168138808], "baseline_config": 1},
    # kernel saturation probe (not a BASELINE config): enough streams to fill every sub-partition
    # 148 SMs x 4 sub-partitions x 8 warps x 32 lanes = 151552 streams
    "saturate_151552x112KiB": {"sizes": [112 << 10] * 151552, "baseline_config": None},
    "tiny": {"sizes": [1 << 20] * 64, "baseline_config": None},
    # BASELINE.json configs[3]: Ollama manifest + 7B GGUF layer blobs (SURVEY.md section 8d sizes: model layer of a
    # typical 7B Q4_0, license, params, config), digest verify sharded by dm_shard_of over the ranks
    # (4 B200 in the config).  One layer dominates: one chain on one GPU, whatever N is.
    "ollama_7b_manifest": {"sizes": [3826793677, 11357, 17, 420], "baseline_config": 3, "routing": "digest"},
    # BASELINE.json configs[4]: blob-size sweep, scaled DOWN and saying so: classes 1 MiB .. 1 GiB in x4 steps
    # (the config's 64 GiB top class is one 14-minute serial chain on any number of GPUs), 2 GiB per class per
    # GPU = 12 GiB per GPU per step (the config: 1 TB over 8 GPUs = 125 GB per GPU) - per-class GB/s in `classes`.
    "size_sweep": {"sizes": [sz for k in range(20, 31, 2) for sz in [1 << k] * ((2 << 30) >> k)], "baseline_config": 4,
                   "classes": [1 << k for k in range(20, 31, 2)],
                   "scaled": "top class 1 GiB instead of 64 GiB (x1/64), 12 GiB per GPU per step instead of 125 GB (x1/10)"},
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _cpu_quota():
    try:
        q, p_ = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(p_)
    except Exception:
        return None


def _cfs_throttle():
    """(nr_throttled, throttled_usec) of this cgroup (CFS bandwidth control), or None.  More runnable threads than the
    CPU quota freeze the WHOLE group - the engine's pump and the CUDA driver threads included - for the rest of each
    100 ms period once the quota is spent; the e2e leg reports how much of that it saw."""
    try:
        kv = dict(ln.split() for ln in open("/sys/fs/cgroup/cpu.stat").read().strip().splitlines())
        return int(kv.get("nr_throttled", 0)), int(kv.get("throttled_usec", 0))
    except Exception:
        return None


def _kernel_for(n):
    """Mirror of streams_per_warp_for() in demodel_b200/csrc/sha256_kernels.cuh (for the report only)."""
    for limit, name in ((296, "deep (1 stream/warp pair)"), (592, "group (2 streams/warp pair)"), (1184, "group (4 streams/warp pair)"),
                        (2368, "group (8 streams/warp pair)"), (4736, "group (16 streams/warp pair)"), (9472, "group (16 streams/warp)")):
        if n <= limit:
            return name
    return "wide (32 streams/warp)"


def _int_issue_roofline(n_streams, hashed_gbs, sm_mhz):
    """The bound that actually binds SHA-256 on sm_100a (DESIGN.md section 5, profiles/r01_ubench_issue_rates.txt):
    the ALU pipe takes one warp-instruction per 2 cycles per sub-partition.  Chip ceiling: >= 1040 ALU-pipe
    instructions per 64-byte block per warp of 32 lanes on 592 sub-partitions.  Few streams: one warp per
    stream needs the round's six rotations and four boolean functions on that pipe whatever is done with the
    additions = 20 cycles per round, 64 rounds per 64 bytes (the shipped round form issues 11: 22 cycles).
    Reported beside the HBM roofline the metric asks for; never raises."""
    try:
        ghz = (sm_mhz or 1965.0) / 1e3
        chip = 592 * ghz * (32 * 64) / (1040 * 2)                 # GB/s
        per_stream = ghz / 20.0                                    # GB/s: 1 byte per round
        peak = min(chip, n_streams * per_stream)
        return {"bound": "int32 ALU-pipe issue", "peak": peak, "achieved": hashed_gbs, "frac": hashed_gbs / peak, "unit": "GB/s hashed",
                "chip_ceiling": chip, "per_stream_ceiling": per_stream, "streams": n_streams, "sm_ghz": ghz}
    except Exception as ex:                                        # reporting only
        return {"error": repr(ex)}


def _numa_bind(local_rank):
    """Opt-in (--numa-bind): pin this process (and every thread it creates later: pump, spill, connection
    workers) to the CPUs of the NUMA node its GPU hangs off, so the pinned ring and the host buffers are
    first-touched there.  Returns a description or None if the topology is not visible."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"gpu_bus": bus, "numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def _layout(sizes):
    offs, pos = [], 0
    for s in sizes:
        offs.append(pos)
        pos += (s + 255) // 256 * 256
    return offs, pos


DUMP_MAX_BLOBS = 1 << 18            # 32 MiB of float32 digests; larger batches are sampled
DUMP_CACHE_BLOBS, DUMP_CACHE_BYTES = 256, 4096


def dump_outputs(out_dir, eng, digests, matched, sizes, blob_ids, cached, prefix=""):
    """What the timed step returned, as float32/float64 .npy files under out_dir, so that two builds run with the
    same arguments (hence the same seeded inputs) can be compared output for output:
      digests.npy      (k, 32) float32  the SHA-256 of each blob, one byte per value
      matched.npy      (k,)    float32  1 where the digest equalled the expected one
      blob_index.npy   (k,)    float64  which synthetic blob each row is (all of them up to DUMP_MAX_BLOBS, else a
                                        fixed seeded sample)
      cache_sample.npy (m,)    float32  bytes read back from the CAS through the hit path (dm_cache_open/read), a
                                        window of up to DUMP_CACHE_BYTES in each of up to DUMP_CACHE_BLOBS blobs;
                                        hash-and-cache mode only
      cache_sample_at.npy (b, 3) float64  (blob index, offset, length) of each window in cache_sample.npy
    At most about 39 MiB in all.  With N > 1 GPUs each rank writes its own set, its names prefixed rank<r>_."""
    import numpy as np
    n = len(sizes)
    rng = np.random.default_rng(SEED)
    rows = np.arange(n) if n <= DUMP_MAX_BLOBS else np.sort(rng.choice(n, DUMP_MAX_BLOBS, replace=False))
    blob_ids = np.asarray(blob_ids, dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)

    def save(name, arr):
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), arr)
    save("digests", np.asarray(digests).reshape(n, 32)[rows].astype(np.float32))
    save("matched", np.asarray(matched)[rows].astype(np.float32))
    save("blob_index", blob_ids[rows])
    if not cached:
        return
    picks = rows if len(rows) <= DUMP_CACHE_BLOBS else np.sort(rng.choice(rows, DUMP_CACHE_BLOBS, replace=False))
    at, parts = [], []
    for r in picks:
        ln = min(DUMP_CACHE_BYTES, int(sizes[r]))
        off = int(rng.integers(0, int(sizes[r]) - ln + 1))
        rid, _ = eng.cache_open(np.asarray(digests)[32 * r:32 * r + 32].tobytes())
        try:
            parts.append(np.frombuffer(eng.cache_read(rid, off, ln), dtype=np.uint8))
        finally:
            eng.cache_close(rid)
        at.append((blob_ids[r], off, ln))
    save("cache_sample", np.concatenate(parts).astype(np.float32) if parts else np.zeros(0, dtype=np.float32))
    save("cache_sample_at", np.asarray(at, dtype=np.float64).reshape(-1, 3))


def _my_blob_indices(n_blobs, rank, world):
    """Disjoint per-rank blob sets chosen by the production router: synthetic
    blobs have no digest before they are hashed, so they are homed by URL hash
    (demodel_b200.shard.owner_of_url), the rule for unknown-digest blobs."""
    from demodel_b200.shard import owner_of_url
    if world == 1:
        return list(range(n_blobs))
    out, k = [], 0
    while len(out) < n_blobs:
        if owner_of_url(f"synthetic://blob/{k}", world) == rank:
            out.append(k)
        k += 1
    return out


def _digest_routed_set(eng, torch, dist, n_total, size_of, rank, world, local, base=0):
    """Fixed blob set routed the production way: the digests of blobs 0..n_total-1 are learned once (each rank
    hashes a 1/world slice, hash-only; the digests are exchanged - setup, outside any timed region), then every rank
    keeps the blobs dm_shard_of(digest, world) gives it.  Returns (indices owned, digests of all, per-rank counts)."""
    import numpy as np
    from demodel_b200.engine import shard_of
    mine_slice = list(range(rank, n_total, world))
    sizes = [size_of(i) for i in mine_slice]
    offs, span = _layout(sizes)
    digs_local = np.zeros((len(mine_slice), 32), dtype=np.uint8)
    if mine_slice:
        buf = torch.empty(max(span, 16), dtype=torch.uint8, device=f"cuda:{local}")
        for j, i in enumerate(mine_slice):
            eng.synth_fill_device(SEED, base + i, 0, buf.data_ptr() + offs[j], sizes[j])
        d, _, _ = eng.ingest_device(buf.data_ptr(), offs, sizes, hash_only=True, raw=True)
        digs_local = d.reshape(-1, 32).copy()
        del buf
    all_digs = np.zeros((n_total, 32), dtype=np.uint8)
    if world > 1:
        per = (n_total + world - 1) // world
        send = torch.zeros((per, 32), dtype=torch.uint8, device=f"cuda:{local}")
        send[:len(mine_slice)] = torch.from_numpy(digs_local).to(send.device)
        got = [torch.zeros_like(send) for _ in range(world)]
        dist.all_gather(got, send)
        for r in range(world):
            idx = list(range(r, n_total, world))
            all_digs[idx] = got[r][:len(idx)].cpu().numpy()
    else:
        all_digs[mine_slice] = digs_local
    owner = [shard_of(all_digs[i].tobytes(), world) for i in range(n_total)]
    counts = [owner.count(r) for r in range(world)]
    return [i for i in range(n_total) if owner[i] == rank], all_digs, counts


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, rank, world):
    """The CPU arm: OpenSSL hash-and-cache loop on all host threads."""
    if rank != 0:
        return
    import numpy as np
    from tests import _oracle
    orc = _oracle.load()
    sizes = WORKLOADS[args.workload]["sizes"]
    ncpu = os.cpu_count() or 1
    threads = min(ncpu, len(sizes))
    quota_threads = min(int(_cpu_quota() or ncpu), len(sizes))
    # bounded sample: whole blobs, at most ~16 GiB so K steps stay within minutes
    budget, take, tot = 16 << 30, 0, 0
    while take < len(sizes) and (take == 0 or tot + sizes[take] <= budget):
        tot += sizes[take]; take += 1
    sizes = sizes[:take]
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    src = np.empty(int(off[-1]), dtype=np.uint8)
    import demodel_b200  # product generator (CPU half), only to make the bytes
    lib = demodel_b200.load()
    import ctypes as C

    def fill(i):
        lib.dm_synth_fill_host(SEED, i, 0, C.c_void_p(src.ctypes.data + int(off[i])), sizes[i])
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(ncpu, 64)) as ex:
        list(ex.map(fill, range(len(sizes))))
    cache = np.empty_like(src)
    total = int(off[-1])
    # give the CPU arm its best thread count (all logical CPUs vs the cgroup quota)
    trial = {}
    for th in sorted({threads, quota_threads}):
        orc.hash_and_cache(src, off, chunk=32768, threads=th, cache=cache)
        trial[th] = orc.hash_and_cache(src, off, chunk=32768, threads=th, cache=cache)[0]
    threads = min(trial, key=trial.get)
    for _ in range(args.warmup):
        orc.hash_and_cache(src, off, chunk=32768, threads=threads, cache=cache)
    t = 0.0
    for _ in range(args.steps):
        secs, digs = orc.hash_and_cache(src, off, chunk=32768, threads=threads, cache=cache)
        t += secs
    gbs = total * args.steps / t / 1e9
    sample = f"{len(sizes)} of {len(WORKLOADS[args.workload]['sizes'])} blobs, {total} B per step, 32 KiB updates + memcpy into an in-memory cache"
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        # same key names as the GPU arm's config for what the two arms share
        "config": {"workload": args.workload, "baseline_config": WORKLOADS[args.workload]["baseline_config"],
                   "blobs_per_gpu": len(WORKLOADS[args.workload]["sizes"]), "bytes_per_gpu_per_step": sum(WORKLOADS[args.workload]["sizes"]),
                   "sampled_blobs": len(sizes), "sampled_bytes_per_step": total, "seed": hex(SEED),
                   "mode": "hash-and-cache (32 KiB EVP_DigestUpdate + memcpy into an in-memory cache)",
                   "note": "OpenSSL EVP_sha256 stand-in for Go crypto/sha256 (no Go toolchain; reference has no such loop)"},
        "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="hf_lfs_256x64MiB")
    ap.add_argument("--kernel", default=None, choices=[None, "wide", "deep"])
    ap.add_argument("--hash-only", action="store_true", help="value leg without the fused CAS copy (1 B/B)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-serve", action="store_true")
    ap.add_argument("--no-probes", action="store_true", help="skip the short many-stream kernel probes")
    ap.add_argument("--e2e-zero-copy", action="store_true")
    ap.add_argument("--ring-mib", type=int, default=1024)
    ap.add_argument("--slab-kib", type=int, default=1024)
    ap.add_argument("--e2e-concurrency", type=int, default=256)
    ap.add_argument("--e2e-threads", type=int, default=0)
    ap.add_argument("--numa-bind", action="store_true", help="pin the process to the GPU's NUMA node (default when N > 1)")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--cas-slack-mib", type=int, default=4096, help="HBM arena beyond one copy of the workload (ring-path bodies, probes)")
    ap.add_argument("--blobs", type=int, default=0, help="override: number of blobs (with --blob-bytes)")
    ap.add_argument("--blob-bytes", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.blobs and args.blob_bytes:
        args.workload = f"custom_{args.blobs}x{args.blob_bytes}"
        WORKLOADS[args.workload] = {"sizes": [args.blob_bytes] * args.blobs, "baseline_config": None}
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # Each rank's connection threads, pump and pinned ring belong on its GPU's NUMA node: at N=8 the e2e
    # leg is bound by host memory traffic (67 GB/s unbound -> 108 GB/s bound, measured); neutral at N=1.
    numa = _numa_bind(local) if (args.numa_bind or (world > 1 and not args.no_numa_bind)) else None
    import numpy as np
    import torch
    import torch.distributed as dist
    import demodel_b200

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback on the hash path)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = WORKLOADS[args.workload]
    routing = wl.get("routing", "url")
    hbm_peak, peak_src = _peaks()
    sizes_all = wl["sizes"]
    if routing == "digest":
        # FIXED blob set (strong scaling): blob i goes to the rank dm_shard_of(digest_i, world) names; a rank may own
        # nothing.  The digests are learned first (setup), as a manifest would have announced them.
        boot = demodel_b200.Engine(device=local, hbm_cas_bytes=256 << 20, ring_bytes=64 << 20)
        mine, all_digs, shard_counts = _digest_routed_set(boot, torch, dist, len(sizes_all), lambda i: sizes_all[i], rank, world, local)
        boot.close()
        sizes = [sizes_all[i] for i in mine]
    else:
        sizes = sizes_all
        mine = _my_blob_indices(len(sizes), rank, world)
        shard_counts = None
    n = len(sizes)
    offs, span = _layout(sizes)
    offs_arr = np.asarray(offs, dtype=np.uint64)      # converted once: no per-step list marshalling
    sizes_arr = np.asarray(sizes, dtype=np.uint64)
    total = sum(sizes)
    job_total = sum(sizes_all) if routing == "digest" else total * world      # bytes the whole job moves per step

    # one copy of the workload (N > 1: 1.5 copies, room for the digest-routed probe's uneven shares) + slack for ring-path bodies
    cas_bytes = 0 if args.hash_only else (span + (64 << 20) if world == 1 else int(1.5 * span) + (64 << 20))
    eng = demodel_b200.Engine(device=local, hbm_cas_bytes=max(cas_bytes, 256 << 20) + (args.cas_slack_mib << 20), ring_bytes=args.ring_mib << 20,
                              slab_bytes=args.slab_kib << 10, max_streams=max(65536, n + 1024))
    dev = torch.empty(max(span, 16), dtype=torch.uint8, device=f"cuda:{local}")
    # blob indices are consecutive per rank only when world == 1; fill one by one otherwise
    if n and mine == list(range(mine[0], mine[0] + n)):
        eng.synth_fill_device_many(SEED, mine[0], dev.data_ptr(), offs, sizes)
    else:
        for i, k in enumerate(mine):
            eng.synth_fill_device(SEED, k, 0, dev.data_ptr() + offs[i], sizes[i])
    torch.cuda.synchronize()

    # ---- value leg: inputs resident in HBM --------------------------------------------
    digs, _, _ = eng.ingest_device(dev.data_ptr(), offs, sizes, hash_only=True, kernel=args.kernel)   # learn the oids
    expect = b"".join(digs)
    expect_arr = np.frombuffer(expect, dtype=np.uint8)

    def step():
        return eng.ingest_device(dev.data_ptr(), offs_arr, sizes_arr, expect=expect, hash_only=args.hash_only,
                                 replace=not args.hash_only, kernel=args.kernel, raw=True)

    for _ in range(args.warmup):
        d, m, _ = step()
        assert np.array_equal(d, expect_arr) and m.all()
    s0 = eng.stats()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    kernel_ms = 0.0
    for _ in range(args.steps):
        d, m, ms = step()
        kernel_ms += ms
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    s1 = eng.stats()
    assert np.array_equal(d, expect_arr) and m.all()
    launches = int(s1["kernel_launches"] - s0["kernel_launches"])
    if args.dump_outputs:                               # before the later legs evict what the timed steps cached
        dump_outputs(args.dump_outputs, eng, d, m, sizes, mine, cached=not args.hash_only,
                     prefix="" if world == 1 else f"rank{rank}_")

    tt = torch.tensor([wall, kernel_ms], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    wall_max, kernel_ms_max = float(tt[0]), float(tt[1])
    value = job_total * args.steps / wall_max / 1e9
    bytes_per_blob_byte = 1 if args.hash_only else 2
    # roofline of the dominant kernel on the busiest rank: its algorithmic bytes / its CUDA-event time
    tb = torch.tensor([float(total)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
    achieved = bytes_per_blob_byte * float(tb[0]) * args.steps / (max(kernel_ms_max, 1e-9) / 1e3) / 1e9

    # spot check against an independent implementation on the host (hashlib), outside the timed region
    import hashlib
    if n:
        probe = min(range(n), key=lambda i: sizes[i])
        host_probe = dev[offs[probe]:offs[probe] + sizes[probe]].cpu().numpy()
        assert hashlib.sha256(host_probe.tobytes()).digest() == digs[probe], "GPU digest differs from hashlib"
    if routing == "digest":                             # the routed digests are the ones the timed steps verified against
        assert [all_digs[i].tobytes() for i in mine] == digs

    # ---- size sweep: each size class on its own (kernel time; inputs and expectations as in the aggregate pass) ----
    classes = None
    if wl.get("classes"):
        classes = []
        for csz in wl["classes"]:
            idx = [i for i in range(n) if sizes[i] == csz]
            if not idx:
                continue
            lo, hi = idx[0], idx[-1] + 1
            exp_c = expect[32 * lo:32 * hi]
            kms = []
            for it in range(2):                          # one untimed pass, one measured (the aggregate leg above is the warm-up proper)
                _, mc, ms_ = eng.ingest_device(dev.data_ptr(), offs_arr[lo:hi], sizes_arr[lo:hi], expect=exp_c, replace=True, raw=True)
                assert mc.all()
                kms.append(ms_)
            tc = torch.tensor([kms[-1]], dtype=torch.float64, device=f"cuda:{local}")
            if world > 1:
                dist.all_reduce(tc, op=dist.ReduceOp.MAX)
            cb = csz * len(idx)
            classes.append({"blob_bytes": csz, "blobs_per_gpu": len(idx), "bytes_per_gpu": cb, "kernel_ms": float(tc[0]),
                            "GBps": cb * world / (float(tc[0]) / 1e3) / 1e9, "kernel": _kernel_for(len(idx)),
                            "hbm_frac": 2 * cb / (float(tc[0]) / 1e3) / 1e9 / hbm_peak})

    # ---- probes: the other kernel shapes at stream counts that fill the chip (kernel time only) ----
    probes = None
    if rank == 0 and not args.no_probes and args.blobs == 0 and routing == "url" and not wl.get("classes"):
        probes = {}
        for name, pn, pbytes in (("wide_151552_streams", 151552, 16384), ("group8_4096_streams", 4096, 524288)):
            po = np.arange(pn, dtype=np.uint64) * np.uint64(pbytes)
            pl = np.full(pn, pbytes, dtype=np.uint64)
            pdev = torch.empty(pn * pbytes, dtype=torch.uint8, device=f"cuda:{local}")
            eng.synth_fill_device_many(SEED, 1 << 20, pdev.data_ptr(), po, pl)
            pd, _, _ = eng.ingest_device(pdev.data_ptr(), po, pl, hash_only=True, raw=True)
            pexp = pd.tobytes()
            kms = []
            for it in range(8):
                _, pm, ms_ = eng.ingest_device(pdev.data_ptr(), po, pl, expect=pexp, replace=True, raw=True)
                assert pm.all()
                if it >= 3:
                    kms.append(ms_)
            k_ms = sum(kms) / len(kms)
            ach = 2 * pn * pbytes / (k_ms / 1e3) / 1e9
            probes[name] = {"streams": pn, "blob_bytes": pbytes, "kernel_ms": k_ms, "hashed_GBps": ach / 2,
                            "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                                         "frac": ach / hbm_peak, "algorithmic_bytes_per_blob_byte": 2},
                            "alu_issue_bound_GBps": 1146.0, "frac_of_alu_bound": ach / 2 / 1146.0}
            import ctypes as _C
            lib_ = demodel_b200.load()
            for i_ in range(pn):                                # drop the probe's blobs from the CAS
                lib_.dm_cache_evict(eng._h, _C.c_char_p(pexp[32 * i_:32 * i_ + 32]))
            del pdev

    # small-blob latency through the stream API: open -> write 4 KiB -> finish (DMA + launch + digest back)
    if probes is not None:
        small = np.random.default_rng(SEED).integers(0, 256, 4096, dtype=np.uint8)
        lat = []
        for it in range(220):
            t0_ = time.perf_counter()
            sid_ = eng.stream_open(None, 4096)
            eng.stream_write(sid_, small)
            d_, _ = eng.stream_finish(sid_)
            lat.append(time.perf_counter() - t0_)
            eng.cache_evict(d_)
        lat = sorted(lat[20:])
        probes["small_blob_latency_us"] = {"p50": 1e6 * lat[len(lat) // 2], "p99": 1e6 * lat[int(len(lat) * 0.99)],
                                          "what": "dm_stream_open + write(4 KiB) + finish, one at a time, via ctypes"}

    # ---- e2e leg: host buffers through the proxy-facing C-ABI ---------------------------
    e2e = None
    if not args.no_e2e:
        hoff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        host = np.empty(int(hoff[-1]), dtype=np.uint8)
        for i in range(n):   # D2H of the same bytes the value leg hashed (setup, untimed)
            host[int(hoff[i]):int(hoff[i + 1])] = dev[offs[i]:offs[i] + sizes[i]].cpu().numpy()
        for d_ in digs:
            eng.cache_evict(d_)
        conc = min(n, args.e2e_concurrency)
        ncpu_eff = int(_cpu_quota() or os.cpu_count() or 1)
        # GOMAXPROCS-style worker threads; half the usable cores measured best (the pump thread, the
        # CUDA driver's threads and the DMA submissions share the same cgroup quota)
        # ... and the ranks of one node share it, so each takes its 1/world share.
        drive_threads = max(1, min(conc, args.e2e_threads or max(1, ncpu_eff // (2 * world))))
        e2e_steps = max(1, min(args.steps, 3))
        for _ in range(1):
            dd, mm, _ = eng.proxy_drive(host, hoff, expect=expect, chunk=32768, concurrency=conc,
                                        nthreads=drive_threads, zero_copy=args.e2e_zero_copy)
            assert dd == digs and all(mm)
            for d_ in digs:
                eng.cache_evict(d_)
        barrier()
        es0 = eng.stats()
        thr0 = _cfs_throttle()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            dd, mm, _ = eng.proxy_drive(host, hoff, expect=expect, chunk=32768, concurrency=conc,
                                        nthreads=drive_threads, zero_copy=args.e2e_zero_copy)
            for d_ in digs:
                eng.cache_evict(d_)
        barrier()
        e_wall = time.perf_counter() - t0
        thr1 = _cfs_throttle()
        assert dd == digs and all(mm)
        es1 = eng.stats()
        # cache-hit path: everything just ingested is served back out to host memory
        serve = None
        if not args.no_serve:
            dd, mm, _ = eng.proxy_drive(host, hoff, expect=expect, chunk=32768, concurrency=conc,
                                        nthreads=drive_threads, zero_copy=args.e2e_zero_copy)
            out = np.empty_like(host)
            eng.proxy_serve(digs[:min(n, 8)], out, hoff[:min(n, 8) + 1], chunk=1 << 20, nthreads=drive_threads)   # warm
            secs = eng.proxy_serve(digs, out, hoff, chunk=1 << 20, nthreads=drive_threads)
            probe_i = n // 2
            if n:
                assert np.array_equal(out[int(hoff[probe_i]):int(hoff[probe_i + 1])], host[int(hoff[probe_i]):int(hoff[probe_i + 1])])
            serve = {"value": total / max(secs, 1e-9) / 1e9, "unit": UNIT, "threads": drive_threads, "read_bytes": 1 << 20,
                     "api": "dm_proxy_serve -> dm_cache_open/read/close"}
            for d_ in digs:
                eng.cache_evict(d_)
            del out
        te = torch.tensor([e_wall], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": job_total * e2e_steps / float(te[0]) / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": total, "d2h_bytes_per_step": 32 * n, "steps": e2e_steps,
               "launches_per_step": (es1["kernel_launches"] - es0["kernel_launches"]) / e2e_steps,
               "kernel_ms_sum_per_step": (es1["kernel_ms"] - es0["kernel_ms"]) / e2e_steps,
               "ring_waits_per_step": (es1["ring_waits"] - es0["ring_waits"]) / e2e_steps,
               "cfs_throttled_ms_per_step": ((thr1[1] - thr0[1]) / 1e3 / e2e_steps) if thr0 and thr1 else None,
               "cfs_throttled_periods_per_step": ((thr1[0] - thr0[0]) / e2e_steps) if thr0 and thr1 else None,
               "hit_serving": serve,
               "api": "dm_proxy_drive -> dm_stream_open/write/flush/finish, 32 KiB pieces, %d concurrent bodies on %d threads%s"
                      % (conc, drive_threads, ", zero-copy ring windows" if args.e2e_zero_copy else "")}
        del host

    # ---- digest-prefix sharding of a FIXED set (N > 1): what the weak-scaling line above cannot show -------------
    # The headline gives every rank exactly n blobs.  Production routes by dm_shard_of(digest): a fixed set of
    # n x N blobs lands unevenly (binomial).  Measured here: per-rank counts, the imbalance, and the whole-set rate
    # with the barrier-to-barrier time of the slowest rank.
    sharding = None
    if world > 1 and routing == "url" and not args.no_probes and args.blobs == 0 and not wl.get("classes") and not args.hash_only:
        for d_ in digs:
            eng.cache_evict(d_)
        del dev
        torch.cuda.empty_cache()
        n_fixed = n * world
        owned, fd, counts = _digest_routed_set(eng, torch, dist, n_fixed, lambda i: sizes[i % n], rank, world, local, base=1 << 24)
        fdev, ready = None, 1.0
        try:                                  # a rank-local failure (its share does not fit) must not leave the others in a collective
            fs = [sizes[i % n] for i in owned]
            fo, fspan = _layout(fs)
            fdev = torch.empty(max(fspan, 16), dtype=torch.uint8, device=f"cuda:{local}")
            for j, i in enumerate(owned):
                eng.synth_fill_device(SEED, (1 << 24) + i, 0, fdev.data_ptr() + fo[j], fs[j])
            fexp = b"".join(fd[i].tobytes() for i in owned)
            fo_a, fs_a = np.asarray(fo, dtype=np.uint64), np.asarray(fs, dtype=np.uint64)
            for _ in range(2):
                _, fm, _ = eng.ingest_device(fdev.data_ptr(), fo_a, fs_a, expect=fexp, replace=True, raw=True)
                assert fm.all()
        except Exception as ex:                # noqa: BLE001
            ready = 0.0
            sharding = {"error": f"rank {rank}: {ex!r}", "blobs_per_rank": counts}
        agree = torch.tensor([ready], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if float(agree[0]) > 0:
            f_steps = max(1, min(args.steps, 3))
            barrier()
            t0 = time.perf_counter()
            fk = 0.0
            for _ in range(f_steps):
                _, fm, ms_ = eng.ingest_device(fdev.data_ptr(), fo_a, fs_a, expect=fexp, replace=True, raw=True)
                fk += ms_
            barrier()
            f_wall = time.perf_counter() - t0
            tf = torch.tensor([f_wall, fk, 1.0 if fm.all() else 0.0], dtype=torch.float64, device=f"cuda:{local}")
            tmin = tf.clone()
            dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            fbytes = sum(sizes[i % n] for i in range(n_fixed))
            sharding = {"mode": "fixed set routed by dm_shard_of(digest, N)", "blobs": n_fixed, "blobs_per_rank": counts,
                        "imbalance_max_over_mean": max(counts) / (n_fixed / world), "steps": f_steps, "all_verified": bool(float(tmin[2]) > 0),
                        "value": fbytes * f_steps / float(tf[0]) / 1e9, "unit": UNIT, "ms_per_step": 1e3 * float(tf[0]) / f_steps,
                        "kernel_ms_per_step_max_rank": float(tf[1]) / f_steps,
                        "note": "warp-per-stream regime: a rank's time is its longest chain, not its blob count, while it holds "
                                "<= 592 streams (one per sub-partition) - the imbalance costs HBM, not time"}
        elif sharding is None:
            sharding = {"error": "another rank could not set up its share", "blobs_per_rank": counts}
        for i in owned:
            eng.cache_evict(fd[i].tobytes())
        del fdev
        dev = torch.empty(16, dtype=torch.uint8, device=f"cuda:{local}")

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only) -----------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from tests import _oracle
        orc = _oracle.load()
        take = 0
        tot = 0
        while take < n and (take == 0 or tot + sizes[take] <= (16 << 30)):
            tot += sizes[take]; take += 1
        coff = np.concatenate([[0], np.cumsum(sizes[:take])]).astype(np.uint64)
        src = np.empty(int(coff[-1]), dtype=np.uint8)
        for i in range(take):
            src[int(coff[i]):int(coff[i + 1])] = dev[offs[i]:offs[i] + sizes[i]].cpu().numpy()
        cache = np.empty_like(src)
        cands = sorted({min(os.cpu_count() or 1, take), min(int(_cpu_quota() or os.cpu_count() or 1), take)})
        best = None
        for threads in cands:                      # give the CPU arm its best thread count
            orc.hash_and_cache(src, coff, chunk=32768, threads=threads, cache=cache)          # warm
            secs, cd = orc.hash_and_cache(src, coff, chunk=32768, threads=threads, cache=cache)
            assert cd == digs[:take], "CPU arm and GPU digests differ"
            if best is None or secs < best[0]:
                best = (secs, threads)
        secs, threads = best
        # BASELINE.md's variant: the cache is a content-addressed file tree on tmpfs instead of memory
        tmpfs_gbs = None
        try:
            import shutil
            import tempfile
            tdir = tempfile.mkdtemp(prefix="dm_cpu_cas_", dir="/dev/shm")
            fsecs, fd_ = orc.hash_and_cache_files(src, coff, tdir, chunk=32768, threads=threads)
            if fsecs > 0 and fd_ == digs[:take]:
                tmpfs_gbs = tot / fsecs / 1e9
            shutil.rmtree(tdir, ignore_errors=True)
        except Exception:
            tmpfs_gbs = None
        secs1, _ = orc.hash_and_cache(src, coff[:2], chunk=32768, threads=1, cache=cache)
        cpu = {"value": tot / secs / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{take} of {n} blobs ({tot} B), OpenSSL EVP_sha256 32 KiB updates + memcpy to an in-memory cache "
                         f"(stand-in for Go crypto/sha256)",
               "single_core_gbs": sizes[0] / secs1 / 1e9, "host_cpus": os.cpu_count(),
               "tmpfs_cas_value": tmpfs_gbs}
        del src, cache

    if rank == 0:
        # roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from an
        # ncu capture of this workload (tools/prof_default.sh writes profiles/roofline_traffic.json).  It is only
        # reported when the capture was taken with the kernel variant that ran here.
        traffic, traffic_src = None, None
        lib_ = demodel_b200.load()
        variant_now = os.environ.get("DM_KERNEL_VARIANT") or f"{lib_.dm_default_kernel_variant(0)},{lib_.dm_default_kernel_variant(1)}"
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath) and not (args.hash_only or args.kernel):
            try:
                ent = json.load(open(tpath)).get(args.workload)
                # the capture is of ONE kernel family: only that half of "wide,deep" has to match what ran
                half = 0 if isinstance(ent, dict) and ent.get("family") == "wide" else 1
                if isinstance(ent, dict) and ent.get("kernel_variant", "").split(",")[half:half + 1] == variant_now.split(",")[half:half + 1]:
                    traffic, traffic_src = ent["bytes"], ent.get("source")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * wall_max / args.steps, "higher_is_better": True, "scaling": "strong" if routing == "digest" else "weak",
            "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": args.workload, "baseline_config": WORKLOADS[args.workload]["baseline_config"],
                       "blobs_per_gpu": n, "bytes_per_gpu_per_step": total, "mode": "hash-only" if args.hash_only else "hash-and-cache (fused CAS copy)",
                       "kernel": args.kernel or _kernel_for(n), "seed": hex(SEED),
                       "l2": "inputs (%.1f GB) larger than L2 (126 MB); no flush needed" % (total / 1e9),
                       "parallelism": (f"shard{world} (fixed set routed by dm_shard_of(digest), no collective)" if routing == "digest"
                                       else f"shard{world} (URL-hash homed, no collective)"),
                       "blobs_per_rank": shard_counts, "scaled": wl.get("scaled"), "job_bytes_per_step": job_total},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel_variant": variant_now, "peak_source": peak_src,
                         "algorithmic_bytes_per_blob_byte": bytes_per_blob_byte, "kernel_ms_per_step": kernel_ms_max / args.steps,
                         "int_issue": _int_issue_roofline(n, achieved / bytes_per_blob_byte, (clocks or {}).get("sm_mhz"))},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "probes": probes,
            "classes": classes, "sharding": sharding,
            "notes": {
                "workload_choice": "BASELINE configs[2] (256 x 64 MiB, 17.18 GB) is the largest single-GPU configuration; "
                                   "configs[1] (4 Llama-3-8B shards, 16.06 GB) is selectable with --workload llama3_8b_shards",
                "configs1_expectation": "SHA-256 chains block to block, so 4 blobs are 4 serial chains: --workload llama3_8b_shards "
                                        "measured 0.2455 GB/s (65.4 s per pass: the 5.0 GB shard at 76.4 MB/s), CPU arm 5.35 GB/s on 4 cores",
                "binding_bound": "integer ALU issue (~1.15 TB/s per B200 for SHA-256), not HBM; see DESIGN.md section 5",
            },
            "host": {"cpus": os.cpu_count(), "cpu_quota": _cpu_quota(), "kernel_variant": os.environ.get("DM_KERNEL_VARIANT"),
                     "numa_bind": numa},
        }
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
