#!/usr/bin/env python
"""bench.py — shuffle write+read GB/s (compress + CRC / verify + decompress) on BASELINE.json's configurations.

  --config 2 (default at --gpus 1): terasort 10 GiB per GPU, 80 maps x 200 partitions = 16,000 shuffle blocks of 671,112 B,
                                    LZ4Block 32 KiB + CRC32C ("terasort 10 GB, 200 partitions, LZ4 + CRC32C, 1xB200"); with
                                    --gpus N every rank owns its own 10 GiB (weak scaling)
  --config 3 (default at --gpus >1): terasort 100 GiB, 800 maps x 2000 partitions = 1.6 M shuffle blocks of 65,520 B (two full
                                    LZ4 blocks + end mark each), block i -> GPU i mod N (strong scaling: the total is fixed).  A
                                    rank keeps one WAVE of <= 200,000 blocks (13 GB) resident and runs ceil(share / wave) passes
                                    per step (SURVEY.md §8d: "stream the dataset in waves and accumulate time")
  --config 4: the SQL-join exchange volume of config 4 — 50 GiB, 80,000 shuffle blocks, Snappy (xerial), split i mod N
  --config 5: Zstandard, shuffle-block size sweep 4 KiB .. 64 MiB on one GPU (value = the 640 KiB point)

One "step" = one write pass (b2s_compress_*: XXH32 + match/parse/emit + framing + CRC32C over the compressed streams) plus
one read pass (b2s_decompress_*: CRC32C verify + decode + XXH32 verify) over the rank's whole share.
  value : uncompressed bytes / (t_write + t_read), inputs and outputs resident in HBM (device API)
  e2e   : the same through the host-pointer C ABI a JVM would call (NUMA-local pinned host arenas; H2D and D2H inside the
          timed region).  Two modes are timed: e2e.serial = one call at a time (round 1's figure), e2e.concurrent = a
          map-side compress call and a reduce-side decompress call in flight together from two task threads (one per lane
          of the ABI, both directions of the PCIe link).  e2e.value is the faster of the two and e2e.mode names it
  roofline : dominant kernel algorithmic bytes (1+r)*U per launch / CUDA-event duration vs measured HBM peak
  cpu_baseline : the reference's CPU arithmetic (liblz4 / libzstd / restated snappy + framing + XXH32 + CRC32C, oracle/), all
                 host cores the cgroup grants, bounded sample of the same data
`--impl reference` times that CPU path alone on the same config (the reference itself is Scala on a JVM, absent here).
`--dump-outputs DIR` writes what the last timed step returned to its caller (rank 0's share) as DIR/<name>.npy, see
dump_outputs(); the inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
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
# one hardware work queue per stream of the library's two lanes (read at CUDA context creation, which torch / NCCL may do
# before b2s_init gets the chance: csrc/api.cu, b2s_init)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

RECORD = 104
LZ4_BLOCK = 32768
# ncu --set full, one launch over 32,768 codec blocks, dram__bytes_read + dram__bytes_write; scaled to the blocks one launch
# of this run processes.  Default pipeline (lz4_match_kernel<12>): profiles/r2z_final.md; B2S_LZ4_PIPE=4
# (lz4_match2_kernel<12>): profiles/r2_compress_generations.md
NCU_TRAFFIC_PER_CODEC_BLOCK = {1: (1.944139e9 + 4.139978e9) / 32768, 4: (1.564307e9 + 2.059700e9) / 32768}
METRIC = "shuffle write+read GB/s (compress+CRC) at 1/2/4/8 B200 vs JVM-LZ4 CPU baseline"
WAVE_BLOCKS_SMALL = 200000   # 65,520-B blocks per resident wave (13.1 GB)
WAVE_BLOCKS_LARGE = 20000    # 671,112-B blocks per resident wave (13.4 GB)
# --dump-outputs: the leading bytes of this many shuffle blocks (a seeded choice) are stored as they left the device; the
# per-block arrays cover every block (<= WAVE_BLOCKS_SMALL of them), so the files stay far below DUMP_LIMIT
DUMP_SAMPLE_BLOCKS = 16
DUMP_SAMPLE_BYTES = 256 << 10
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, c, w, r, d_cmp, d_out):
    """Writes the last timed wave's results as float64 (per-block integers) and float32 (bytes) .npy files:
    compressed_{offsets,lengths,crc32c,status} from the compress call, decompressed_{offsets,lengths,status} from the
    decompress call, decompressed_crc32c over every decoded block, and for the blocks in sample_blocks the first
    DUMP_SAMPLE_BYTES of each compressed stream and of each decoded block, concatenated (compressed_sample,
    decompressed_sample)."""
    n = w["dst_len"].size
    pick = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SAMPLE_BLOCKS), replace=False))

    def sample(d_base, offs, lens):
        parts = []
        for i in pick:
            part = np.empty(min(int(lens[i]), DUMP_SAMPLE_BYTES), dtype=np.uint8)
            if part.size:
                c.dev_memcpy(part.ctypes.data, d_base + int(offs[i]), part.size, 2)
            parts.append(part)
        return np.concatenate(parts).astype(np.float32)

    arrays = {
        "compressed_offsets": w["dst_off"], "compressed_lengths": w["dst_len"], "compressed_crc32c": w["checksums"],
        "compressed_status": w["status"], "decompressed_offsets": r["dst_off"], "decompressed_lengths": r["dst_len"],
        "decompressed_status": r["status"],
        "decompressed_crc32c": c.checksum_dev(c.CHECKSUM_CRC32C, d_out, r["dst_off"], r["dst_len"]),
        "sample_blocks": pick,
    }
    arrays = {k: np.asarray(v).astype(np.float64) for k, v in arrays.items()}
    arrays["compressed_sample"] = sample(d_cmp, w["dst_off"], w["dst_len"])
    arrays["decompressed_sample"] = sample(d_out, r["dst_off"], r["dst_len"])
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, "outputs to dump (%d B) exceed %d B" % (total, DUMP_LIMIT)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def usable_cores():
    """host threads this process may really use: the affinity mask, capped by the cgroup CPU quota (a 1-GPU lease of the
    128-thread host gets cpu.max = 16 cores: round 1 printed 128 there and measured 14 cores' worth)"""
    n = len(os.sched_getaffinity(0))
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    cores = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return cores, n, quota


def bind_process_to_gpu_node(gpu_index):
    """sched_setaffinity + set_mempolicy(MPOL_PREFERRED) to the NUMA node of GPU `gpu_index` (sysfs; no libnuma).
    Returns the node or None when the topology cannot be read (then nothing is changed)."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout
        bdf = None
        for line in q.strip().splitlines():
            idx, b = [x.strip() for x in line.split(",")]
            if int(idx) == gpu_index:
                bdf = b.lower()
        if bdf is None:
            return None
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        import ctypes
        libc = ctypes.CDLL(None, use_errno=True)
        mask = (ctypes.c_ulong * 16)()
        mask[node // 64] = 1 << (node % 64)
        libc.syscall(238, 1, mask, 1025)  # SYS_set_mempolicy, MPOL_PREFERRED
        return node
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


CPU_NOTES = {
    "lz4": "oracle framing/XXH32/CRC32C + liblz4.so.1 LZ4_compress_default/LZ4_decompress_fast (the native routines "
           "lz4-java's JNI path calls); no JVM stream wrappers / JNI => upper bound on the reference",
    "snappy": "oracle xerial framing + restated raw-Snappy compressor/decompressor + CRC32C (snappy-java's native side is "
              "absent here); no JVM stream wrappers / JNI",
    "zstd": "libzstd.so.1 ZSTD_compress level 3 / ZSTD_decompress (what zstd-jni executes; BASELINE config 5's level) + "
            "CRC32C; no JVM stream wrappers / JNI => upper bound on the reference",
}


def cpu_arm(oracle, codec, sample, block_bytes, threads, repeats=1):
    """reference CPU arithmetic on `sample` (numpy uint8): returns (GB/s write+read, detail)"""
    best = None
    for _ in range(repeats):
        r = oracle.baseline_run_codec(codec, sample, block_bytes, LZ4_BLOCK, oracle.CRC32C, threads=threads, level=3)
        if r["rc"] != 0:
            raise RuntimeError("CPU baseline reported %d errors" % r["errors"])
        t = r["write_s"] + r["read_s"]
        if best is None or t < best[0]:
            best = (t, r)
    t, r = best
    return r["bytes"] / t / 1e9, r


def plan(args, world):
    """-> dict(codec, records_per_block, blocks (per rank, per wave), waves, scaling, workload text)"""
    cfg = args.config if args.config else (2 if world == 1 else 3)
    if cfg == 2:
        rpb, codec, total_blocks = 6453, "lz4", 16000 * world
        per_rank, scaling = 16000, "weak"
        what = "config 2: terasort 10.00 GiB per GPU, 80 maps x 200 partitions = 16,000 shuffle blocks x 671,112 B"
    elif cfg == 3:
        rpb, codec, total_blocks = 630, "lz4", 1600000
        per_rank, scaling = -(-total_blocks // world), "strong"
        what = ("config 3: terasort 100 GiB, 800 maps x 2000 partitions = 1,600,000 shuffle blocks x 65,520 B "
                "(2 full LZ4 blocks + end mark each), block i -> GPU i mod %d" % world)
    elif cfg == 4:
        rpb, codec, total_blocks = 6453, "snappy", 80000
        per_rank, scaling = -(-total_blocks // world), "strong"
        what = ("config 4: SQL-join exchange volume 50 GiB, 400 maps x 200 partitions = 80,000 shuffle blocks x 671,112 B "
                "(terasort-shaped records; the UnsafeRow shape is covered by tests/test_gpu_snappy.py), block i -> GPU i mod %d" % world)
    else:
        raise SystemExit("--config 5 is the block-size sweep: run tools/zstd_sweep.py (bench.py --config 5 forwards to it)")
    if args.codec:
        codec = args.codec
    if args.records_per_block:
        rpb = args.records_per_block
    if args.blocks:
        per_rank = args.blocks
    cap = WAVE_BLOCKS_SMALL if rpb * RECORD < 200000 else WAVE_BLOCKS_LARGE
    waves = max(1, -(-per_rank // cap))
    wave_blocks = -(-per_rank // waves)
    return {"config": cfg, "codec": codec, "rpb": rpb, "wave_blocks": wave_blocks, "waves": waves, "scaling": scaling,
            "what": what, "per_rank": wave_blocks * waves}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3, 4, 5],
                    help="BASELINE.json configuration; 0 = config 2 at --gpus 1, config 3 at --gpus > 1")
    ap.add_argument("--blocks", type=int, default=int(os.environ.get("B2S_BENCH_BLOCKS", 0)),
                    help="shuffle blocks per GPU (overrides the configuration; smaller only for quick checks)")
    ap.add_argument("--records-per-block", type=int, default=0,
                    help="104-byte records per shuffle block (overrides the configuration): 6453 = 671,112 B, 630 = 65,520 B")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample-bytes", type=int, default=4 << 30, help="uncompressed bytes of the CPU arm's sample per step")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--codec", default="", choices=["", "lz4", "snappy", "zstd"],
                    help="override the configuration's codec (lz4 = LZ4Block, snappy = xerial, zstd)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.config == 5):
        ap.error("--dump-outputs needs the device-resident B200 arm (--impl b200, --config 2/3/4)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.config == 5:
        if rank == 0:
            os.execv(sys.executable, [sys.executable, os.path.join(ROOT, "tools", "zstd_sweep.py"), "--bench-line"])
        return 0
    steps, warmup = args.steps, max(args.warmup, 3)
    P = plan(args, world)
    codec_name, rpb, n, waves = P["codec"], P["rpb"], P["wave_blocks"], P["waves"]
    block_bytes = rpb * RECORD
    wave_bytes = n * block_bytes
    rank_bytes = wave_bytes * waves
    codec_desc = {"lz4": "lz4 (LZ4Block, blockSize 32 KiB)", "snappy": "snappy (xerial framing, blockSize 32 KiB)",
                  "zstd": "zstd (frames of 32 KiB blocks)"}[codec_name]
    workload = "%s; %s + CRC32C" % (P["what"], codec_desc)
    config = {"workload": workload, "baseline_config": P["config"], "codec": codec_desc,
              "checksum": "CRC32C over compressed bytes", "blocks_per_gpu": n * waves, "block_bytes": block_bytes,
              "waves_per_step": waves, "wave_blocks": n,
              "l2_policy": "every pass streams >= 6 GB per GPU, far larger than the 126 MB L2",
              "sharding": "block i -> GPU i mod N (each rank owns its blocks; no collective on the data path)"}
    if waves > 1:
        config["waves_note"] = ("a rank's share (%.1f GB) is processed as %d passes over one resident wave of %d blocks"
                                % (rank_bytes / 1e9, waves, n))

    from oracle import oracle  # CPU baseline legs only (never on the GPU product path)

    # ------------------------------------------------------------------ reference arm: CPU only
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads, aff, quota = usable_cores()
        sample_blocks = max(1, min(args.cpu_sample_bytes // block_bytes, n))
        sample = oracle.gen_terasort(0, sample_blocks * rpb)
        cpu_arm(oracle, codec_name, sample[: min(sample_blocks, 200) * block_bytes], block_bytes, threads)
        vals, t0 = [], time.perf_counter()
        for _ in range(steps):
            v, detail = cpu_arm(oracle, codec_name, sample, block_bytes, threads)
            vals.append(v)
        wall = time.perf_counter() - t0
        value = sample.size * steps / sum(sample.size / (v * 1e9) for v in vals) / 1e9
        sample_desc = "%d of %d shuffle blocks (%.2f GiB) per step, same generator/seed" % (
            sample_blocks, n * waves * world, sample.size / 2**30)
        line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warmup, "ms_per_step": round(wall / steps * 1e3, 3), "higher_is_better": True,
                "scaling": P["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": round(value, 3), "unit": "GB/s", "cores": threads,
                                 "affinity_threads": aff, "cgroup_cpu_quota": quota, "kind": "port", "sample": sample_desc,
                                 "note": CPU_NOTES[codec_name],
                                 "compressed_ratio": round(detail["compressed_bytes"] / detail["bytes"], 4)},
                "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    # NUMA first, before torch / CUDA / NCCL create their helper threads and arenas: the whole rank process (its threads,
    # page cache, pinned staging) lives on the socket its GPU hangs off.  GPUs 0-3 / 4-7 sit on different sockets of the
    # 8-GPU hosts; round 1's ranks floated over both and the host-staged path lost half its scaling to cross-socket
    # traffic (VERDICT round 1).  The C ABI repeats the placement for its own allocations (b2s_bind_thread_to_device).
    early_numa = bind_process_to_gpu_node(local_rank) if os.environ.get("B2S_NUMA", "1") != "0" else None
    import torch

    torch.cuda.set_device(local_rank)
    import spark_s3_shuffle_b200 as pkg

    rk = pkg.ranks.Ranks(backend="nccl", device=torch.device("cuda", local_rank))  # barrier + max-over-ranks only
    c = pkg.capi
    c.init(1 << local_rank)
    L = c.load()
    # the rank's host threads and pinned arenas live on the socket its GPU hangs off (SURVEY.md §8e)
    numa_node = c.bind_thread_to_device(0)
    barrier, max_over_ranks = rk.barrier, rk.max_over_ranks

    CODEC = {"lz4": c.CODEC_LZ4BLOCK, "snappy": c.CODEC_SNAPPY_XERIAL, "zstd": c.CODEC_ZSTD}[codec_name]
    LEVEL = 3 if codec_name == "zstd" else 0
    cmp_cap = int(c.compress_bound(CODEC, LZ4_BLOCK, block_bytes)) * n
    d_src, d_cmp, d_out = c.dev_alloc(wave_bytes), c.dev_alloc(cmp_cap), c.dev_alloc(wave_bytes)
    c.gen_terasort_dev(d_src, rank * n * rpb, n * rpb, 42)
    off = np.arange(n, dtype=np.uint64) * block_bytes
    ln = np.full(n, block_bytes, dtype=np.uint64)
    sb = np.arange(n + 1, dtype=np.uint32)

    kt = {"write_kernel_ms": [], "read_kernel_ms": [], "compress_ms": [], "decompress_ms": [], "match_ms": [],
          "match_launches": []}

    def wave_device(record):
        w = c.compress_dev(CODEC, d_src, off, ln, d_cmp, cmp_cap, LZ4_BLOCK, c.CHECKSUM_CRC32C, level=LEVEL)
        tw = c.last_timing()
        r = c.decompress_dev(CODEC, d_cmp, w["dst_off"], w["dst_len"], d_out, wave_bytes, c.CHECKSUM_CRC32C, sb,
                             w["dst_len"], w["checksums"])
        tr = c.last_timing()
        if record:
            kt["write_kernel_ms"].append(tw["kernel_ms"]); kt["compress_ms"].append(tw["top_kernel_ms"])
            kt["match_ms"].append(tw["dominant_ms"]); kt["match_launches"].append(tw["dominant_launches"])
            kt["read_kernel_ms"].append(tr["kernel_ms"]); kt["decompress_ms"].append(tr["top_kernel_ms"])
        return w, r

    def step_device(record):
        for _ in range(waves):
            w, r = wave_device(record)
        return w, r

    want = c.checksum_dev(c.CHECKSUM_CRC32C, d_src, off, ln)
    for _ in range(warmup):
        w, r = step_device(False)
    assert not w["status"].any() and not r["status"].any() and r["total"] == wave_bytes, "device round trip failed"
    got = c.checksum_dev(c.CHECKSUM_CRC32C, d_out, off, ln)
    assert (got == want).all(), "decode(encode(x)) != x"
    ratio = w["total"] / wave_bytes

    sampler = ClockSampler(local_rank)
    launches0 = L.b2s_total_kernel_launches()
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    c.mark(0)                      # CUDA events on the library's own stream (every call is synchronous)
    for _ in range(steps):
        w, r = step_device(True)
    c.mark(1)
    dev_elapsed = c.marks_elapsed_ms() * 1e-3
    barrier()
    wall = time.perf_counter() - t0
    elapsed = max_over_ranks(max(dev_elapsed, 0.0) if dev_elapsed > 0.5 * wall else wall)
    clocks = sampler.stop()
    launches = L.b2s_total_kernel_launches() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, c, w, r, d_cmp, d_out)
    ms_per_step = elapsed / steps * 1e3
    value = world * rank_bytes / (elapsed / steps) / 1e9

    comp_ms = statistics.mean(kt["compress_ms"])          # per wave
    match_ms = statistics.mean(kt["match_ms"])
    match_launches = max(1, int(statistics.mean(kt["match_launches"])))
    dec_ms = statistics.mean(kt["decompress_ms"])
    peak, peak_src = measured_peak()
    pipe = int(os.environ.get("B2S_LZ4_PIPE", "1"))
    dom_kernel = "lz4_match2_kernel<12>" if pipe != 1 else "lz4_match_kernel<12>"
    # dominant kernel = the match kernel (phase A of the compressor; largest share in profiles/*launches*.csv).
    # achieved = SURVEY §8(d)'s write-step figure (1+r) x the input bytes one launch processes / its launch duration.
    step_alg = (1.0 + ratio) * wave_bytes                  # compress step reads U, writes C (= decompress step mirrored)
    alg_bytes = step_alg / match_launches
    achieved = alg_bytes / (match_ms / match_launches * 1e-3) / 1e9
    codec_blocks_per_launch = n * -(-block_bytes // LZ4_BLOCK) / match_launches
    roofline = {"bound": "hbm", "kernel": dom_kernel, "achieved": round(achieved, 2), "peak": peak,
                "unit": "GB/s", "frac": round(achieved / peak, 5),
                "traffic": (int(NCU_TRAFFIC_PER_CODEC_BLOCK[pipe] * codec_blocks_per_launch)
                            if pipe in NCU_TRAFFIC_PER_CODEC_BLOCK and codec_name == "lz4" else None),
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg_bytes), "avg_launch_ms": round(match_ms / match_launches, 4),
                "launches_per_wave": match_launches,
                "compress_step": {"kernels": "match + parse + scan + emit (what one fused kernel would do)",
                                  "algorithmic_bytes": int(step_alg), "ms": round(comp_ms, 3),
                                  "achieved": round(step_alg / (comp_ms * 1e-3) / 1e9, 2),
                                  "frac": round(step_alg / (comp_ms * 1e-3) / 1e9 / peak, 5)},
                "decompress_step": {"kernels": "tokens + copy", "algorithmic_bytes": int(step_alg),
                                    "ms": round(dec_ms, 3), "achieved": round(step_alg / (dec_ms * 1e-3) / 1e9, 2),
                                    "frac": round(step_alg / (dec_ms * 1e-3) / 1e9 / peak, 5)},
                "note": "LZ77 coding is issue/latency-bound byte-stream work; traffic (ncu dram bytes per launch, "
                        "profiles/) exceeds the algorithmic bytes by the per-position off[] table handed to the parse kernel"}
    kernels = {"per": "wave", "compress_ms": round(comp_ms, 3), "match_ms": round(match_ms, 3), "decompress_ms": round(dec_ms, 3),
               "write_pass_kernels_ms": round(statistics.mean(kt["write_kernel_ms"]), 3),
               "read_pass_kernels_ms": round(statistics.mean(kt["read_kernel_ms"]), 3),
               "compress_GBps_uncompressed": round(wave_bytes / comp_ms / 1e6, 2),
               "decompress_GBps_uncompressed": round(wave_bytes / dec_ms / 1e6, 2)}

    # ------------------------------------------------------------------ e2e through the host-pointer C ABI
    e2e = None
    if not args.no_e2e:
        # pinned host arenas (NUMA-local: b2s_host_alloc places them next to the rank's GPU): source, compressed (write
        # side), compressed copy (read side's input while the write side overwrites its own), decoded
        def alloc():
            bufs = []
            try:
                for nbytes in (wave_bytes, cmp_cap, cmp_cap, wave_bytes):
                    bufs.append(c.HostBuffer(nbytes))
                return bufs
            except Exception:
                for hb in bufs:
                    hb.free()
                return None

        bufs = alloc()
        if max_over_ranks(0.0 if bufs is not None else 1.0) > 0:
            if bufs is not None:
                for hb in bufs:
                    hb.free()
            e2e = {"value": None, "unit": "GB/s", "error": "pinned host memory for the end-to-end leg could not be allocated"}
        else:
            h_src, h_cmp, h_cmp_in, h_out = bufs
            c.dev_memcpy(h_src.ptr, d_src, wave_bytes, 2)
            for p in (d_src, d_cmp, d_out):
                c.dev_free(p)
            d_src = d_cmp = d_out = None

            def write_pass():
                w = c.compress_packed(CODEC, h_src.array, off, ln, h_cmp.array, LZ4_BLOCK, c.CHECKSUM_CRC32C, level=LEVEL)
                return w, c.last_timing()

            def read_pass(w, src):
                r = c.decompress_packed(CODEC, src.array, w["dst_off"], w["dst_len"], h_out.array,
                                        c.CHECKSUM_CRC32C, sb, w["dst_len"], w["checksums"])
                return r, c.last_timing()

            w, tw = write_pass()   # warm-up (allocates slot buffers)
            r, tr = read_pass(w, h_cmp)
            assert not w["status"].any() and not r["status"].any() and r["total"] == wave_bytes
            for i in (0, n // 2, n - 1):
                a = h_src.array[i * block_bytes:(i + 1) * block_bytes]
                b = h_out.array[int(r["dst_off"][i]):int(r["dst_off"][i]) + block_bytes]
                assert np.array_equal(a, b), "e2e round trip mismatch"
            h_cmp_in.array[: w["total"]] = h_cmp.array[: w["total"]]
            w0 = w

            # ---- serial: one call at a time (write pass, then read pass)
            write_pass(); read_pass(w0, h_cmp)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                for _ in range(waves):
                    w, tw = write_pass()
                    r, tr = read_pass(w, h_cmp)
            barrier()
            s_elapsed = max_over_ranks(time.perf_counter() - t0)
            s_val = world * rank_bytes / (s_elapsed / args.e2e_steps) / 1e9
            serial = {"value": round(s_val, 3), "ms_per_step": round(s_elapsed / args.e2e_steps * 1e3, 2),
                      "write_ms": round(tw["total_ms"], 2), "read_ms": round(tr["total_ms"], 2),
                      "write_sums_ms": {k: round(tw[k], 1) for k in ("h2d_ms", "kernel_ms", "d2h_ms")},
                      "read_sums_ms": {k: round(tr[k], 1) for k in ("h2d_ms", "kernel_ms", "d2h_ms")}}

            # ---- write || read: two task threads, one per lane of the ABI (map-side compress of this wave while the
            # reduce side decodes the previous wave's output), both directions of the link busy
            errs = []
            tms = {}

            def writer():
                try:
                    c.bind_thread_to_device(0)
                    for _ in range(args.e2e_steps * waves):
                        ww, t = write_pass()
                        assert not ww["status"].any()
                    tms["w"] = t
                except Exception as ex:  # noqa: BLE001
                    errs.append(repr(ex))

            def reader():
                try:
                    c.bind_thread_to_device(0)
                    for _ in range(args.e2e_steps * waves):
                        rr, t = read_pass(w0, h_cmp_in)
                        assert not rr["status"].any() and rr["total"] == wave_bytes
                    tms["r"] = t
                except Exception as ex:  # noqa: BLE001
                    errs.append(repr(ex))

            barrier()
            t0 = time.perf_counter()
            ths = [threading.Thread(target=writer), threading.Thread(target=reader)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
            barrier()
            c_elapsed = max_over_ranks(time.perf_counter() - t0)
            if errs:
                raise RuntimeError("concurrent e2e leg failed: %s" % errs)
            c_val = world * rank_bytes / (c_elapsed / args.e2e_steps) / 1e9
            tw2, tr2 = tms["w"], tms["r"]
            concurrent = {"value": round(c_val, 3), "ms_per_step": round(c_elapsed / args.e2e_steps * 1e3, 2),
                          "write_ms": round(tw2["total_ms"], 2), "read_ms": round(tr2["total_ms"], 2),
                          "write_sums_ms": {k: round(tw2[k], 1) for k in ("h2d_ms", "kernel_ms", "d2h_ms")},
                          "read_sums_ms": {k: round(tr2[k], 1) for k in ("h2d_ms", "kernel_ms", "d2h_ms")}}
            # headline = the faster of the two ways of driving the ABI, named (DESIGN.md §5c: the two lanes remove the lock,
            # but one FIFO copy queue per direction keeps the duplex gain away for now)
            best_serial = s_val >= c_val
            e2e = {"value": round(max(s_val, c_val), 3), "unit": "GB/s",
                   "mode": ("serial: one C-ABI call at a time (write pass, then read pass)" if best_serial else
                            "write || read: a compress call and a decompress call in flight together from two task "
                            "threads (one per ABI lane)"),
                   "h2d_bytes_per_step": int((tw2["h2d_bytes"] + tr2["h2d_bytes"]) * waves),
                   "d2h_bytes_per_step": int((tw2["d2h_bytes"] + tr2["d2h_bytes"]) * waves),
                   "ms_per_step": round((s_elapsed if best_serial else c_elapsed) / args.e2e_steps * 1e3, 2),
                   "steps": args.e2e_steps, "blocks_per_gpu": n * waves, "numa_node": numa_node,
                   "process_bound_to_node": early_numa, "serial": serial, "concurrent": concurrent,
                   "api": "b2s_compress_packed + b2s_decompress_packed on NUMA-local pinned host arenas (b2s_host_alloc)"}
            if world == 1 and n >= 200:
                # what ONE Spark task hands over: a map task's 200 partitions (commitAllPartitions), a reduce task's
                # 80 map outputs (S3ShuffleReader.read) — latency of a single synchronous C-ABI call, median of 5
                tws, trs = [], []
                for _ in range(6):
                    t = time.perf_counter()
                    w1 = c.compress_packed(CODEC, h_src.array, off[:200], ln[:200], h_cmp.array, LZ4_BLOCK,
                                           c.CHECKSUM_CRC32C, level=LEVEL)
                    tws.append(time.perf_counter() - t)
                    t = time.perf_counter()
                    r1 = c.decompress_packed(CODEC, h_cmp.array, w1["dst_off"][:80], w1["dst_len"][:80], h_out.array,
                                             c.CHECKSUM_CRC32C, sb[:81], w1["dst_len"][:80], w1["checksums"][:80])
                    trs.append(time.perf_counter() - t)
                    assert not w1["status"].any() and not r1["status"].any()
                tw1, tr1 = statistics.median(tws[1:]), statistics.median(trs[1:])
                e2e["task_sized_calls"] = {
                    "map_task": {"blocks": 200, "uncompressed_MB": round(200 * block_bytes / 1e6, 1),
                                 "ms": round(tw1 * 1e3, 2), "GBps": round(200 * block_bytes / tw1 / 1e9, 2)},
                    "reduce_task": {"blocks": 80, "uncompressed_MB": round(80 * block_bytes / 1e6, 1),
                                    "ms": round(tr1 * 1e3, 2), "GBps": round(80 * block_bytes / tr1 / 1e9, 2)}}

    # ------------------------------------------------------------------ CPU baseline beside it (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads, aff, quota = usable_cores()
        sample_blocks = max(1, min(args.cpu_sample_bytes // block_bytes, n))
        sample = oracle.gen_terasort(0, sample_blocks * rpb)
        cpu_arm(oracle, codec_name, sample[: min(200, sample_blocks) * block_bytes], block_bytes, threads)
        v, detail = cpu_arm(oracle, codec_name, sample, block_bytes, threads, repeats=2)
        v1, _ = cpu_arm(oracle, codec_name, sample[: min(64, sample_blocks) * block_bytes], block_bytes, 1)
        cpu = {"value": round(v, 3), "unit": "GB/s", "cores": threads, "affinity_threads": aff, "cgroup_cpu_quota": quota,
               "kind": "port",
               "sample": "%d of %d shuffle blocks (%.2f GiB), same generator/seed, best of 2" % (
                   sample_blocks, n * waves, sample.size / 2**30),
               "single_core_GBps": round(v1, 3),
               "note": CPU_NOTES[codec_name]}

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": steps,
                "warmup": warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": P["scaling"],
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "compressed_ratio": round(ratio, 4), "gpu_launches": int(launches), "clocks": clocks,
                "roofline": roofline, "kernels": kernels}
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    rk.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
